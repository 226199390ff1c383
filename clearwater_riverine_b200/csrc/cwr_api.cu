// C ABI (include/cwr.h) over the sm_100a kernels in cwr_kernels.cuh.
// Host logic only: buffers, per-step parameter block, launch order, the solver driver loop.
#include "../../include/cwr.h"

#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <string>
#include <vector>

#include "cwr_kernels.cuh"
#include "cwr_small.cuh"
#include "cwr_topology.h"

using namespace cwr;

static thread_local std::string g_create_error;

struct cwr_handle {
    int device = 0;
    cudaStream_t stream = nullptr;
    cwr_options opt{};
    Topology topo;
    int n = 0, F = 0, E = 0, K = 0, T = 0, G = 0;
    int C = 0;                       // hydro slices resident
    int KC = 1, VEC = 1;             // lanes per row, columns per lane
    int SKC = 1, SVEC = 1;           // the same for the preconditioner sweeps (128-bit lanes of the sweep type)
    int m_steps = 1;                 // sweeps of the preconditioner + 1 (1 = diagonal scaling only)
    bool sweep_f32 = true;           // preconditioner sweeps (and p^, s^) in fp32
    bool gauss_seidel = false;       // multicolour Gauss-Seidel sweeps instead of Jacobi steps
    bool hint_done = false;          // the colours have been aligned with the flow (or it is too late to)
    int grid_sweep = 0, grid_gs = 0;
    int32_t* d_color_ptr = nullptr;
    bool dc = false;                 // defect-correction solver (options.solver = 2) instead of BiCGSTAB
    bool dc_fixed = false;           // ... with a fixed number of sweeps per cycle (precond_steps given) instead of the device-side plan
    bool strips = false;             // neighbour-synchronised sweep kernel: one strip of rows per CTA (precond_sync = 2, 3)
    bool pipelined = false;          // ... software-pipelined across the synchronisation (k_gs_strip, precond_sync = 3)
    bool tma = false;                // ... with a TMA-fed operand ring and register gathers: fp32 sweeps, K = 16, ELL width 4, one rank
                                     // (k_gs_tma, precond_sync = 4)
    int gs_debug = 0;                // CWR_GS_DEBUG (development)
    int strip_cap = 0;               // rows of a (strip, colour) the sweep kernel takes in one pass
    int n_strips = 0;
    int32_t *d_strip_cptr = nullptr, *d_strip_nptr = nullptr, *d_strip_nbr = nullptr; size_t strip_nbr_cap = 0;
    unsigned long long* d_strip_flag = nullptr;
    uint8_t* d_strip_peers = nullptr;
    unsigned long long gs_seq = 0;   // launches of the sweep kernel so far (epoch of the strip flags)
    int last_cycles = 0;             // cycles of the previous defect-correction solve (launch-ahead prediction)
    double* cur_x = nullptr;         // c[t+1] slot of the step being solved (the iterate)
    int64_t sweeps_total = 0, fallbacks = 0;
    // sparse real-cell overrides of one step, flattened for k_patch_rows
    std::vector<long long> ov_idx; std::vector<double> ov_val;
    long long* d_ov_idx = nullptr; double* d_ov_val = nullptr; size_t ov_cap = 0;
    // domain decomposition (world == 1: plain single-GPU handle)
    int rank = 0, world = 1;
    bool attached = false;           // peers' slabs are mapped (cwr_dd_attach)
    char* d_slab = nullptr; size_t slab_bytes = 0;     // symmetric slab: DdCtl | p^ | s^ | tmp | state slots
    uint8_t* d_send_mask = nullptr; int32_t* d_send_rows = nullptr;
    std::vector<void*> peer_maps;    // cudaIpcOpenMemHandle results to close
    std::vector<int32_t> f1_ref, f2_ref;   // the caller's connectivity (kept for the flow-aligned recolouring)
    int last_iters = 0;              // iterations of the previous solve (launch-ahead prediction)
    bool small_path = false;         // one-CTA-per-column in-kernel solve (small meshes)
    bool tiny = false;               // ... entirely on chip (k_solve_tiny: matrix in shared memory, Gauss-Seidel sweeps)
    int tiny_rpt = 1;                // rows per thread of k_solve_tiny
    int max_optin_smem = 0;
    bool pdl = false;                // small-mesh path: the step's kernels are launched with programmatic stream serialization
    int chip_ns = 0;                 // > 0: k_solve_chip with this many colour slots per thread (ELL width 4, colours of <= 256 rows)
    bool in_run = false;             // inside cwr_run: the small path does not synchronise per step
    SmallStats* d_stats = nullptr; SmallStats* h_stats = nullptr;
    int num_sms = 148, grid_rows = 0, grid_edges = 0, grid_b = 0, max_grid = 0, grid_spmm = 0, grid_at = 0, grid_xrp = 0;
    DeviceModel M{};
    // device buffers
    int32_t *d_ell_col = nullptr, *d_ell_code = nullptr, *d_f1p = nullptr, *d_f2p = nullptr;
    int32_t *d_bcell = nullptr, *d_bptr = nullptr, *d_bedge = nullptr, *d_eperm = nullptr, *d_einv = nullptr;
    int32_t *d_new_of_old = nullptr, *d_old_of_new = nullptr, *d_f1 = nullptr, *d_f2 = nullptr;
    float *d_adv = nullptr, *d_velg = nullptr, *d_flowg = nullptr, *d_vol = nullptr;   // (C,E), (C,E_g), (C,E_g), (C,n)
    double* d_cdiff = nullptr;                                    // (C,E)
    double* d_bc = nullptr;                                       // (T,G,K)
    double* d_state = nullptr;                                    // (S,n,K)
    double* d_dist = nullptr;                                     // (E) reference order
    void* d_stage = nullptr; size_t stage_bytes = 0;
    // second stream for uploads that overlap the device->host copies of the previous step (cwr_prefetch_hydro_raw)
    cudaStream_t up_stream = nullptr; cudaEvent_t compute_mark = nullptr;
    std::vector<cudaEvent_t> up_done; std::vector<uint8_t> up_pending;     // per hydro slot: a prefetched slice is on its way
    void* d_stage_up = nullptr; size_t stage_up_bytes = 0;
    // asynchronous outputs (cwr_fetch_async): c[t+1] and the mass fluxes of a step are gathered into one of two staging
    // slots on the compute stream and copied to the host on a third stream while the next step runs
    cudaStream_t out_stream = nullptr; cudaEvent_t ev_extract[2] = {nullptr, nullptr}, ev_copied[2] = {nullptr, nullptr};
    double* d_out[2] = {nullptr, nullptr}; size_t out_bytes[2] = {0, 0}; int out_next = 0; bool out_pending[2] = {false, false};
    StepParams* d_sp = nullptr;
    // cwr_run on the small-mesh path: the parameters of every step of the run are uploaded at once and a step's kernels are
    // given their element (no k_set_step launch per step)
    StepParams* d_sp_ring = nullptr; size_t sp_ring_cap = 0; std::vector<StepParams> sp_host;
    const StepParams* sp_ready = nullptr;      // != nullptr inside such a run: the device copy of the current step's parameters
    HostMirror* h_mirror = nullptr; HostMirror* d_mirror = nullptr;   // page-locked, mapped into the device (k_mirror)
    SolverCtl* h_ctl = nullptr;                                   // = &h_mirror->ctl
    double* h_sc = nullptr; int* h_flags = nullptr;               // = h_mirror->sc, flags
    int n_state_slots = 0;
    std::vector<double> dt;
    std::vector<int> slot_time;
    std::vector<std::vector<double>> initial_row;                 // per constituent (F)
    std::vector<uint8_t> inputs_set;
    std::vector<std::map<int, std::vector<std::pair<int32_t, double>>>> real_overrides;   // [k][t] -> (device cell, value)
    int computed_upto = 0;           // c[t] valid for t <= computed_upto
    int flux_step = -1;              // step whose mass fluxes are on the device
    int lhs_step = -1;
    bool have_geometry = false;
    int64_t launches = 0, iterations = 0;
    // first-order kinetics (cwr_set_kinetics): the reacting constituents in topological order and their yields; k_react runs
    // in every step while kin_on.  The buffers are allocated by the first call and kept (the reaction mass is a running sum).
    bool kin_on = false;
    int kin_steps = 0, kin_temp_k = -1, kin_grid_max = 0;   // kin_grid_max: resident CTAs of k_react (partials sized for it)
    double kin_temp_c = 20.0;
    KinStep* d_kin_steps = nullptr; KinYield* d_kin_yields = nullptr; KinState* d_kin_state = nullptr; double* d_kin_partials = nullptr;
    // sources and exchange (cwr_set_kinetics_sources): the listed columns in ascending order; kin_src_o2: one is kind 1
    int kin_srcs = 0, kin_src_o2 = 0;
    KinSrc* d_kin_srcs = nullptr;
    // what cwr_set_kinetics_limits validates against: the decay rates and yields of the kinetics set last, the step of
    // each decaying column and the list position of each source column (-1: none)
    std::vector<double> kin_decay_h, kin_yields_h, kin_source_h, kin_exchange_h;
    std::vector<int> kin_step_of, kin_src_of;
    // Monod factors (cwr_set_kinetics_limits): kin_facs entries, grouped per process by d_kin_fptr (n_steps + n_src + 1)
    int kin_facs = 0;
    KinFac* d_kin_facs = nullptr; int* d_kin_fptr = nullptr;
    // depth-scaled processes (cwr_set_kinetics_depth): flags per process (n_steps + n_src, numbered as d_kin_fptr; bit 0 the
    // decay or source, bit 1 the exchange), the plan areas in reference numbering (kin_area_h, F) and per device row
    // (d_kin_area, n; uploaded again when the ordering is rebuilt); k_react<true, true> runs while kin_depth, with the
    // all-zero d_kin_fptr0 when there are no factors
    bool kin_depth = false;
    double kin_min_depth = 0.0;
    std::vector<double> kin_area_h;
    double* d_kin_area = nullptr; int* d_kin_dflag = nullptr; int* d_kin_fptr0 = nullptr;
    // time-varying forcing (cwr_set_kinetics_forcing): the (n, T) series (d_kin_force, room for 1 + 4K of them, allocated
    // by the first call) and the series row of every forced parameter (d_kin_fmap, 1 + n_steps + 3 n_src, see k_react);
    // the kForced instantiations of k_react run while kin_forced.  kin_kind_h: the equilibrium kind of every column
    bool kin_forced = false;
    double* d_kin_force = nullptr; int* d_kin_fmap = nullptr;
    std::vector<int> kin_kind_h;
    // optional per-kernel-family timing with CUDA events on the handle's stream (bench.py roofline)
    bool profiling = false;
    std::vector<cudaEvent_t> ev_pool;
    std::vector<int> ev_family;
    size_t ev_used = 0;
    double fam_ms[CWR_PROFILE_FAMILIES] = {0};
    int64_t fam_count[CWR_PROFILE_FAMILIES] = {0};
    std::string err;
    std::vector<void*> allocs;
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t _e = (call);                                                                   \
        if (_e != cudaSuccess) {                                                                   \
            h->err = std::string(#call) + ": " + cudaGetErrorString(_e);                           \
            return CWR_ECUDA;                                                                      \
        }                                                                                          \
    } while (0)

#define FAIL(code, msg) do { h->err = (msg); return (code); } while (0)

template <typename T>
static cudaError_t dalloc(cwr_handle* h, T** p, size_t count) {
    *p = nullptr;
    if (count == 0) count = 1;
    cudaError_t e = cudaMalloc((void**)p, count * sizeof(T));
    if (e == cudaSuccess) h->allocs.push_back(*p);
    return e;
}

template <typename T>
static cudaError_t upload(cwr_handle* h, T** p, const std::vector<T>& v) {
    cudaError_t e = dalloc(h, p, v.size());
    if (e != cudaSuccess) return e;
    if (!v.empty()) e = cudaMemcpyAsync(*p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream);
    return e;
}

// profiling: an event is recorded before every kernel of a step; the time between two consecutive
// events is attributed to the kernel family launched after the first one.
static inline void mark(cwr_handle* h, int family) {
    if (!h->profiling) return;
    if (h->ev_used == h->ev_pool.size()) {
        cudaEvent_t e;
        if (cudaEventCreate(&e) != cudaSuccess) return;
        h->ev_pool.push_back(e);
        h->ev_family.push_back(0);
    }
    h->ev_family[h->ev_used] = family;
    cudaEventRecord(h->ev_pool[h->ev_used++], h->stream);
}

static void flush_profile(cwr_handle* h) {
    if (!h->profiling || h->ev_used == 0) return;
    mark(h, -1);
    cudaEventSynchronize(h->ev_pool[h->ev_used - 1]);
    for (size_t i = 0; i + 1 < h->ev_used; ++i) {
        const int f = h->ev_family[i];
        if (f < 0 || f >= CWR_PROFILE_FAMILIES) continue;
        float ms = 0.f;
        if (cudaEventElapsedTime(&ms, h->ev_pool[i], h->ev_pool[i + 1]) == cudaSuccess) {
            h->fam_ms[f] += ms;
            h->fam_count[f] += 1;
        }
    }
    h->ev_used = 0;
}

static inline int grid_for(int64_t items, int per_block, int max_grid) {
    int64_t g = (items + per_block - 1) / per_block;
    return (int)std::max<int64_t>(1, std::min<int64_t>(g, max_grid));
}

// (rows, K) interleaved device array -> (K, n) in reference order (k_extract_all: gather + transpose)
static inline void launch_extract(cwr_handle* h, double* out, const double* src, const int32_t* perm, int n, size_t stride_k) {
    const size_t smem = (size_t)kXposeRows * (h->K + 1) * sizeof(double);
    k_extract_all<<<grid_for(n, kXposeRows, h->max_grid), kThreads, smem, h->stream>>>(out, src, perm, n, h->K, stride_k);
    h->launches += 1;
}

static int ensure_stage(cwr_handle* h, size_t bytes) {
    if (bytes <= h->stage_bytes) return CWR_OK;
    if (h->d_stage) { CK(cudaStreamSynchronize(h->stream)); CK(cudaFree(h->d_stage)); h->d_stage = nullptr; h->stage_bytes = 0; }
    CK(cudaMalloc(&h->d_stage, bytes));
    h->stage_bytes = bytes;
    return CWR_OK;
}

#define KC_CASES(...)                          \
    switch (h->KC) {                           \
        case 1: { constexpr int KC = 1; __VA_ARGS__; break; }   \
        case 2: { constexpr int KC = 2; __VA_ARGS__; break; }   \
        case 4: { constexpr int KC = 4; __VA_ARGS__; break; }   \
        case 8: { constexpr int KC = 8; __VA_ARGS__; break; }   \
        case 16: { constexpr int KC = 16; __VA_ARGS__; break; } \
        default: { constexpr int KC = 32; __VA_ARGS__; break; } \
    }
// binds constexpr KC (lanes per row) and VEC (columns per lane) for the handle's K
#define KC_DISPATCH(KCV, ...)                                           \
    if (h->VEC == 2) { constexpr int VEC = 2; KC_CASES(__VA_ARGS__) }   \
    else { constexpr int VEC = 1; KC_CASES(__VA_ARGS__) }

// ---- preconditioner ---------------------------------------------------------------------------------
// binds ST (sweep type), SKC, SVEC for the handle
#define SWEEP_KC_CASES(...)                    \
    switch (h->SKC) {                          \
        case 1: { constexpr int SKC = 1; __VA_ARGS__; break; }   \
        case 2: { constexpr int SKC = 2; __VA_ARGS__; break; }   \
        case 4: { constexpr int SKC = 4; __VA_ARGS__; break; }   \
        case 8: { constexpr int SKC = 8; __VA_ARGS__; break; }   \
        case 16: { constexpr int SKC = 16; __VA_ARGS__; break; } \
        default: { constexpr int SKC = 32; __VA_ARGS__; break; } \
    }
#define SWEEP_DISPATCH(...)                                                                   \
    if (h->sweep_f32) {                                                                       \
        using ST = float;                                                                     \
        if (h->SVEC == 4) { constexpr int SVEC = 4; SWEEP_KC_CASES(__VA_ARGS__) }             \
        else if (h->SVEC == 2) { constexpr int SVEC = 2; SWEEP_KC_CASES(__VA_ARGS__) }        \
        else { constexpr int SVEC = 1; SWEEP_KC_CASES(__VA_ARGS__) }                          \
    } else {                                                                                  \
        using ST = double;                                                                    \
        if (h->SVEC == 2) { constexpr int SVEC = 2; SWEEP_KC_CASES(__VA_ARGS__) }             \
        else { constexpr int SVEC = 1; SWEEP_KC_CASES(__VA_ARGS__) }                          \
    }
// binds RPT (rows per thread) and W4 (ELL width 4) for k_solve_tiny
#define TINY_RPT_CASES(...)                                        \
    switch (h->tiny_rpt) {                                         \
        case 1: { constexpr int RPT = 1; __VA_ARGS__; break; }     \
        case 2: { constexpr int RPT = 2; __VA_ARGS__; break; }     \
        case 3: case 4: { constexpr int RPT = 4; __VA_ARGS__; break; }     \
        case 5: case 6: { constexpr int RPT = 6; __VA_ARGS__; break; }     \
        default: { constexpr int RPT = 8; __VA_ARGS__; break; }    \
    }
#define TINY_DISPATCH(...)                                                     \
    if (h->topo.W == 4) { constexpr bool W4 = true; TINY_RPT_CASES(__VA_ARGS__) } \
    else { constexpr bool W4 = false; TINY_RPT_CASES(__VA_ARGS__) }
// binds PT: the type of the preconditioned vectors p^ / s^ the products and the update kernel read
#define PT_DISPATCH(...)                                                                      \
    if (h->m_steps > 1 && h->sweep_f32) { using PT = float; KC_DISPATCH(h->KC, __VA_ARGS__) } \
    else { using PT = double; KC_DISPATCH(h->KC, __VA_ARGS__) }

// k_gs_strip exists for 16-byte packs of the sweep type only
template <typename ST, int SKC, int SVEC>
static cudaError_t gs3_prepare(int* occ) {
    if constexpr (sizeof(ST) * SVEC == 16) {
        cudaError_t e = cudaFuncSetAttribute(k_gs_strip<ST, SKC, SVEC>, cudaFuncAttributeMaxDynamicSharedMemorySize, gs3_smem_bytes<ST>());
        if (e != cudaSuccess) return e;
        return cudaOccupancyMaxActiveBlocksPerMultiprocessor(occ, k_gs_strip<ST, SKC, SVEC>, kGsThreads, gs3_smem_bytes<ST>());
    } else { *occ = 0; return cudaSuccess; }
}
template <typename ST, int SKC, int SVEC>
static cudaError_t gs3_launch(int grid, void** args, cudaStream_t stream) {
    if constexpr (sizeof(ST) * SVEC == 16)
        return cudaLaunchCooperativeKernel((const void*)k_gs_strip<ST, SKC, SVEC>, dim3(grid), dim3(kGsThreads), args, gs3_smem_bytes<ST>(), stream);
    else return cudaErrorInvalidValue;
}

// copy the (re)built topology into the device arrays allocated by create_impl (sizes do not depend on
// the ordering)
template <typename T>
static cudaError_t put(cwr_handle* h, T* d, const std::vector<T>& v) {
    return v.empty() ? cudaSuccess : cudaMemcpyAsync(d, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice, h->stream);
}

// the plan areas of cwr_set_kinetics_depth in the device order (stream-ordered; pageable source)
static int upload_kin_area(cwr_handle* h) {
    std::vector<double> a(h->n);
    for (int i = 0; i < h->n; ++i) a[i] = h->kin_area_h[h->topo.old_of_new[i]];
    CK(cudaMemcpyAsync(h->d_kin_area, a.data(), a.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    return CWR_OK;
}

static int upload_topology(cwr_handle* h) {
    const Topology& tp = h->topo;
    CK(put(h, h->d_ell_col, tp.ell_col)); CK(put(h, h->d_ell_code, tp.ell_code));
    CK(put(h, h->d_f1p, tp.f1p)); CK(put(h, h->d_f2p, tp.f2p));
    CK(put(h, h->d_bcell, tp.bcell)); CK(put(h, h->d_bptr, tp.bptr)); CK(put(h, h->d_bedge, tp.bedge));
    CK(put(h, h->d_eperm, tp.eperm));
    std::vector<int32_t> einv(tp.E);
    for (int ep = 0; ep < tp.E; ++ep) einv[tp.eperm[ep]] = ep;
    CK(put(h, h->d_einv, einv));
    CK(put(h, h->d_new_of_old, tp.new_of_old)); CK(put(h, h->d_old_of_new, tp.old_of_new));
    CK(put(h, h->d_color_ptr, tp.color_ptr));
    CK(put(h, h->d_send_mask, tp.send_mask)); CK(put(h, h->d_send_rows, tp.send_rows));
    if (h->strips) {
        CK(put(h, h->d_strip_cptr, tp.strip_cptr)); CK(put(h, h->d_strip_nptr, tp.strip_nptr));
        if (tp.strip_nbr.size() > h->strip_nbr_cap) {          // the neighbour lists depend on the ordering
            CK(cudaStreamSynchronize(h->stream));
            if (h->d_strip_nbr) CK(cudaFree(h->d_strip_nbr));
            h->d_strip_nbr = nullptr;
            h->strip_nbr_cap = tp.strip_nbr.size() + tp.strip_nbr.size() / 4 + 16;
            CK(cudaMalloc((void**)&h->d_strip_nbr, h->strip_nbr_cap * sizeof(int32_t)));
        }
        CK(put(h, h->d_strip_nbr, tp.strip_nbr));
        CK(put(h, h->d_strip_peers, tp.strip_peers));
    }
    if (!h->kin_area_h.empty()) {
        const int rc = upload_kin_area(h);
        if (rc) return rc;
    }
    CK(cudaStreamSynchronize(h->stream));
    return CWR_OK;
}

// the part of the (re)built topology this rank owns
static void set_owned_ranges(cwr_handle* h) {
    const Topology& tp = h->topo;
    DeviceModel& M = h->M;
    const int r = h->rank;
    M.row_lo = tp.part_ptr[r]; M.row_hi = tp.part_ptr[r + 1];
    M.ie_lo = tp.iedge_ptr[r]; M.ie_hi = tp.iedge_ptr[r + 1];
    M.ge_lo = tp.gedge_ptr[r]; M.ge_hi = tp.gedge_ptr[r + 1];
    M.b_lo = tp.bcell_ptr[r]; M.b_hi = tp.bcell_ptr[r + 1];
    M.n_colors = tp.n_colors;
    M.color_ptr = h->d_color_ptr + (size_t)r * (tp.n_colors + 1);
    M.strip_cptr = h->d_strip_cptr; M.strip_nptr = h->d_strip_nptr; M.strip_nbr = h->d_strip_nbr; M.strip_peers = h->d_strip_peers;
    // one rank: the flags of its strips; several: the flags of ALL strips in the symmetric slab (the ranks that read rows of
    // a strip hold a mirror of its flag, written by the strip's owner over NVLink)
    M.strip_flag = h->world > 1 ? reinterpret_cast<unsigned long long*>(h->d_slab + kDdFlagOffset) : h->d_strip_flag;
    M.n_strips = h->strips ? h->n_strips : 0; M.strip0 = r * M.n_strips;
    unsigned nbr = 0;
    for (int32_t j = tp.send_ptr[r]; j < tp.send_ptr[r + 1]; ++j) nbr |= tp.send_mask[tp.send_rows[j]];
    M.nbr_mask = nbr;        // symmetric: whoever reads my rows owns rows I read
    M.send_rows = h->d_send_rows + tp.send_ptr[r];
    M.n_send = tp.send_ptr[r + 1] - tp.send_ptr[r];
    M.halo_per_sweep = h->opt.dd_halo_per_colour ? 0 : 1;
}

// Launch of a kernel of the small-mesh step chain: with programmatic stream serialization when h->pdl (every kernel
// launched through here starts with pdl_enter()).
template <typename... KArgs, typename... Args>
static cudaError_t launch_chain(cwr_handle* h, void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, Args&&... args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = h->stream;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = h->pdl ? 1 : 0;
    return cudaLaunchKernelEx(&cfg, kern, std::forward<Args>(args)...);
}

// k_solve_chip (one row of every colour per thread) where the colours allow it: ELL width 4, at most 14 colours of at most
// 256 rows, everything in shared memory.  CWR_TINY_KERNEL=1 keeps k_solve_tiny (for comparisons).
static void choose_chip(cwr_handle* h) {
    const Topology& tp = h->topo;
    h->chip_ns = 0;
    if (!h->tiny) return;
    const char* ev = std::getenv("CWR_TINY_KERNEL");
    if (ev && std::atoi(ev) == 1) return;
    if (tp.W != 4 || tp.n_colors < 1 || tp.n_colors > 14) return;
    int widest = 0;
    for (int c = 0; c < tp.n_colors; ++c) widest = std::max(widest, tp.color_ptr[c + 1] - tp.color_ptr[c]);
    const int ns = tp.n_colors <= 8 ? 8 : (tp.n_colors <= 12 ? 12 : 14);
    if (widest > kChipThreads || chip_smem_bytes(tp.n, ns) + kTinyStaticSmem > (size_t)h->max_optin_smem) return;
    h->chip_ns = ns;
}

// Gauss-Seidel colours follow the flow: the first hydrodynamic slices the caller uploads give the
// direction (time mean of the face flows over the call's slices).  Only possible while nothing that
// depends on the cell order is on the device yet (no inputs, no hydro slices, no steps).
static int align_colours_with_flow(cwr_handle* h, const float* flow, int nt) {
    if (!(h->gauss_seidel || h->tiny) || h->hint_done) return CWR_OK;
    h->hint_done = true;
    for (uint8_t s : h->inputs_set) if (s) return CWR_OK;
    const int E = h->E;
    std::vector<double> mean(E, 0.0);
    const int stride = std::max(1, nt / 32);
    for (int s = 0; s < nt; s += stride)
        for (int e = 0; e < E; ++e) { const float q = flow[(size_t)s * E + e]; if (q == q) mean[e] += q; }
    std::vector<float> hint(E);
    for (int e = 0; e < E; ++e) hint[e] = (float)mean[e];
    Topology t2;
    std::string terr = build_topology(h->n, h->F, E, h->f1_ref.data(), h->f2_ref.data(), h->opt.reorder != 0,
                                      h->opt.precond_colors, hint.data(), h->world, t2, h->strips ? h->n_strips : 0, h->strip_cap);
    if (!terr.empty()) FAIL(CWR_EINVAL, terr);
    if (h->tma && t2.max_strip_nbr > 31) return CWR_OK;      // (a strip of an RCM band has two or three neighbours)
    if (t2.W != h->topo.W || t2.color_ptr.size() != h->topo.color_ptr.size()) return CWR_OK;   // cannot happen: same graph
    if (h->attached) return CWR_OK;                 // peers already rely on the current ownership
    h->topo = std::move(t2);
    choose_chip(h);
    int rc = upload_topology(h);                    // (may move the strip neighbour list)
    set_owned_ranges(h);
    return rc;
}

// domain decomposition: this rank's boundary rows of a slab vector -> the ranks that read them, followed
// by the halo barrier (k_halo_push).  No-op on a single rank.
template <typename T>
static int halo_push(cwr_handle* h, T* vec) {
    if (h->world == 1) return CWR_OK;
    if (!h->attached) FAIL(CWR_EINVAL, "domain-decomposed handle: call cwr_dd_attach before stepping");
    const Topology& tp = h->topo;
    const int n_send = tp.send_ptr[h->rank + 1] - tp.send_ptr[h->rank];
    const int g = grid_for((int64_t)std::max(1, n_send) * h->K, kThreads, 64);
    k_halo_push<T><<<g, kThreads, 0, h->stream>>>(h->M, vec, h->d_send_rows + tp.send_ptr[h->rank], n_send);
    h->launches += 1;
    return CWR_OK;
}

extern "C" {

int cwr_default_options(cwr_options* o) {
    if (!o) return CWR_EINVAL;
    std::memset(o, 0, sizeof(*o));
    o->rtol = 1e-13;
    o->max_iter = 500;
    o->reorder = 1;
    o->keep_history = 1;
    o->hydro_capacity = 0;
    o->mass_flux = 1;
    o->solver_path = 0;
    o->solver = 0;
    o->check_every = 1;
    o->precond_steps = 0;
    o->precond_precision = 32;
    o->precond_sweep = 1;
    o->precond_colors = 0;
    o->precond_sync = 0;
    return CWR_OK;
}

const char* cwr_last_error(const cwr_handle* h) { return h ? h->err.c_str() : g_create_error.c_str(); }

void cwr_destroy(cwr_handle* h) {
    if (!h) return;
    cudaSetDevice(h->device);
    if (h->stream) cudaStreamSynchronize(h->stream);
    if (h->up_stream) { cudaStreamSynchronize(h->up_stream); cudaStreamDestroy(h->up_stream); }
    for (cudaEvent_t e : h->up_done) if (e) cudaEventDestroy(e);
    if (h->compute_mark) cudaEventDestroy(h->compute_mark);
    if (h->d_stage_up) cudaFree(h->d_stage_up);
    if (h->out_stream) { cudaStreamSynchronize(h->out_stream); cudaStreamDestroy(h->out_stream); }
    for (int i = 0; i < 2; ++i) {
        if (h->ev_extract[i]) cudaEventDestroy(h->ev_extract[i]);
        if (h->ev_copied[i]) cudaEventDestroy(h->ev_copied[i]);
        if (h->d_out[i]) cudaFree(h->d_out[i]);
    }
    if (h->d_strip_nbr) cudaFree(h->d_strip_nbr);
    if (h->d_ov_idx) cudaFree(h->d_ov_idx);
    if (h->d_sp_ring) cudaFree(h->d_sp_ring);
    if (h->d_ov_val) cudaFree(h->d_ov_val);
    for (void* p : h->peer_maps) cudaIpcCloseMemHandle(p);
    for (cudaEvent_t e : h->ev_pool) cudaEventDestroy(e);
    for (void* p : h->allocs) cudaFree(p);
    if (h->d_stage) cudaFree(h->d_stage);
    if (h->h_mirror) cudaFreeHost(h->h_mirror);
    if (h->h_stats) cudaFreeHost(h->h_stats);
    if (h->stream) cudaStreamDestroy(h->stream);
    delete h;
}

static int create_impl(cwr_handle* h, int device, int n_real, int n_face, int n_edge, int n_time, int n_const,
                       const int32_t* f1, const int32_t* f2, double D, const cwr_options* opt, const float* flow_hint) {
    if (!f1 || !f2) FAIL(CWR_EINVAL, "f1/f2 must not be NULL");
    if (n_time < 2) FAIL(CWR_EINVAL, "n_time must be >= 2");
    if (n_const < 1 || n_const > kMaxK) FAIL(CWR_EINVAL, "n_const must be in [1, 128]");
    if (opt) h->opt = *opt; else cwr_default_options(&h->opt);
    if (!(h->opt.rtol > 0)) h->opt.rtol = 1e-13;
    if (h->opt.max_iter <= 0) h->opt.max_iter = 500;
    if (h->opt.check_every <= 0) h->opt.check_every = 1;
    const bool small = h->opt.solver_path == 2 || (h->opt.solver_path == 0 && n_real <= 32768);
    // tiny meshes (<= 4096 cells, the Ohio River model): the whole solve on chip with Gauss-Seidel sweeps
    const bool tiny = small && h->opt.precond_sweep == 1 && h->opt.precond_steps != 1 && n_real <= kTinyThreads * kTinyMaxRows;
    // auto: 5 Gauss-Seidel sweeps per application on large meshes (about two BiCGSTAB iterations per step on the
    // 1M x 16 benchmark; with the half-step exit, 5..11 sweeps all land within a few % of each other), 8 on chip
    // (Ohio-shaped mesh, k_solve_chip: 4 / 6 / 8 / 10 sweeps per application 0.077 / 0.074 / 0.072 / 0.077 ms per step),
    // 7 Jacobi steps
    const bool steps_given = h->opt.precond_steps > 0;
    if (h->opt.precond_steps <= 0) h->opt.precond_steps = h->opt.precond_sweep == 1 ? (tiny ? 9 : (!small ? 6 : 8)) : 8;
    h->m_steps = std::min(h->opt.precond_steps, 64);
    if (h->opt.precond_precision != 64) h->opt.precond_precision = 32;
    h->sweep_f32 = h->opt.precond_precision == 32;
    // solver path: small meshes run the whole solve of a column inside one CTA (cwr_small.cuh)
    h->small_path = small;
    h->pdl = small && !std::getenv("CWR_NO_PDL");
    h->world = std::max(1, h->opt.dd_world); h->rank = h->opt.dd_rank;
    if (h->world > kMaxRanks || h->rank < 0 || h->rank >= h->world) FAIL(CWR_EINVAL, "dd_rank / dd_world out of range (at most 8 ranks)");
    if (h->world > 1 && (small || h->m_steps < 2))
        FAIL(CWR_EINVAL, "domain decomposition needs the multi-CTA solver path (solver_path = 1) and precond_steps >= 2");
    h->tiny = tiny;
    h->gauss_seidel = h->opt.precond_sweep == 1 && !h->small_path && h->m_steps > 1;
    if (h->opt.precond_sweep != 0 && h->opt.precond_sweep != 1) FAIL(CWR_EINVAL, "precond_sweep must be 0 (Jacobi steps) or 1 (Gauss-Seidel sweeps)");
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (ndev == 0) FAIL(CWR_ECUDA, "no CUDA device: this library has no CPU fallback");
    if (device < 0 || device >= ndev) FAIL(CWR_EINVAL, "device index out of range");
    h->device = device;
    CK(cudaSetDevice(device));
    CK(cudaStreamCreateWithFlags(&h->stream, cudaStreamNonBlocking));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    h->num_sms = prop.multiProcessorCount;
    {   // lanes per row / columns per lane (128-bit packs), for the fp64 vectors and for the sweep type
        const int K = n_const;
        h->VEC = (K % 2 == 0) ? 2 : 1;
        int kc = 1;
        while (kc * h->VEC < K && kc < 32) kc <<= 1;
        h->KC = kc;
        const int vmax = h->sweep_f32 ? 4 : 2;
        int sv = vmax;
        while (sv > 1 && K % sv != 0) sv >>= 1;
        int skc = 1;
        while (skc * sv < K && skc < 32) skc <<= 1;
        h->SVEC = sv; h->SKC = skc;
    }
    // solver: defect correction with the sweeps themselves where they are Gauss-Seidel sweeps, else BiCGSTAB
    if (h->opt.solver != 1 && h->opt.solver != 2) h->opt.solver = h->gauss_seidel ? 2 : 1;
    h->dc = h->opt.solver == 2 && !h->small_path && h->m_steps > 1;
    h->dc_fixed = h->dc && steps_given;
    if (h->opt.solver == 2 && !h->dc) h->opt.solver = 1;
    // sweep kernel: one strip of rows per resident CTA, synchronised with its neighbour strips only
    if (h->opt.precond_sync < 1 || h->opt.precond_sync > 4) h->opt.precond_sync = h->opt.dd_halo_per_colour ? 1 : 4;
    if (h->opt.precond_sync != 1 && h->opt.dd_halo_per_colour)
        FAIL(CWR_EINVAL, "dd_halo_per_colour needs the grid-barrier sweep kernel (precond_sync = 1)");
    h->strips = h->gauss_seidel && h->opt.precond_sync >= 2;
    h->pipelined = h->gauss_seidel && h->opt.precond_sync >= 3 && (h->sweep_f32 ? 4 : 8) * h->SVEC == 16 && std::max(1, h->opt.dd_world) == 1;
    if (h->gauss_seidel && h->opt.precond_sync >= 3 && !h->pipelined) h->opt.precond_sync = 2;     // packs narrower than 16 bytes / several ranks
    // k_gs_tma: fp32 sweeps, 4 lanes x 16 bytes per row, one rank (ELL width 4 is checked once the topology is known)
    h->tma = h->pipelined && h->opt.precond_sync == 4 && h->sweep_f32 && h->SKC == 4 && h->SVEC == 4 && n_const == 16 &&
             std::max(1, h->opt.dd_world) == 1;
    if (h->pipelined && !h->tma) h->opt.precond_sync = 3;
    if (h->gauss_seidel) {
        int occ_gs = 0, coop = 0;
        if (h->pipelined) {
            cudaError_t e = cudaSuccess;
            SWEEP_DISPATCH(e = gs3_prepare<ST, SKC, SVEC>(&occ_gs));
            CK(e);
            if (h->tma) {
                int occ_tma = 0;
                CK(cudaFuncSetAttribute(k_gs_tma<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTmaSmemBytes));
                CK(cudaFuncSetAttribute(k_gs_tma<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kTmaSmemBytes));
                CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_tma, k_gs_tma<false>, kGsThreads, kTmaSmemBytes));
                if (const char* e = getenv("CWR_GS_DEBUG")) h->gs_debug = atoi(e);
                occ_gs = std::min(occ_gs, occ_tma);       // either kernel may run on these strips
            }
        } else if (h->strips) {
            SWEEP_DISPATCH(cudaFuncSetAttribute(k_precond_gs<ST, SKC, SVEC, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGsSmemBytes));
            SWEEP_DISPATCH(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_gs, k_precond_gs<ST, SKC, SVEC, true>, kGsThreads, kGsSmemBytes));
        } else {
            SWEEP_DISPATCH(cudaFuncSetAttribute(k_precond_gs<ST, SKC, SVEC, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kGsSmemBytes));
            SWEEP_DISPATCH(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_gs, k_precond_gs<ST, SKC, SVEC, false>, kGsThreads, kGsSmemBytes));
        }
        cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, device);
        if (!coop || occ_gs < 1) FAIL(CWR_ECUDA, "cooperative launch not available: use precond_sweep = 0");
        h->grid_gs = h->num_sms * occ_gs;      // every CTA resident: the kernel synchronises between CTAs
        // a strip needs rows of every colour for every lane group to be worth a CTA: small meshes get fewer strips
        const int rows_rank = n_real / std::max(1, h->opt.dd_world);
        h->n_strips = std::max(1, std::min(h->grid_gs, rows_rank / 512));
        if (h->strips) h->grid_gs = h->n_strips;
        if (h->strips) h->strip_cap = kGsRows * (kGsThreads / h->SKC);
    }
    if (h->opt.precond_colors <= 0 && h->strips) {
        // one colour of a strip = one pass of the CTA: kGsRows rows per lane group (the pipelined rows of k_precond_gs)
        const double rows_strip = (double)n_real / std::max(1, h->opt.dd_world) / h->n_strips;
        const int per_pass = h->strip_cap;          // (build_topology moves the rows a colour would hold beyond one pass)
        h->opt.precond_colors = (int)std::min(48.0, std::max(8.0, std::ceil(rows_strip * 1.1 / per_pass)));
    }
    if (h->opt.precond_colors <= 0) {
        // auto: a colour should move ~20 MB (well above the ~4 us a grid barrier + gather latency cost):
        // bytes per row of one sweep = indices + values + three vectors in the sweep type
        const double bytes = (double)n_real / std::max(1, h->opt.dd_world) * (32.0 + 3.0 * n_const * (h->sweep_f32 ? 4 : 8));
        // (a colour's barrier also waits for the neighbour ranks of a domain decomposition: ~10 us, so 40 MB there)
        h->opt.precond_colors = (int)std::lround(std::min(48.0, std::max(8.0, bytes / (h->opt.dd_world > 1 ? 40e6 : 20e6))));
        // on chip a colour costs a CTA barrier: 12 measured best on the Ohio-shaped mesh; one or two more where that lets
        // every colour fit one pass of k_solve_chip (256 rows)
        if (tiny) h->opt.precond_colors = std::max(12, std::min(14, (int)std::ceil(n_real * 1.03 / kChipThreads)));
    }
    if (tiny && !h->strips) h->strip_cap = kChipThreads;      // colours balanced towards <= 256 rows (build_topology)
    h->opt.precond_colors = std::min(h->opt.precond_colors, 64);

    h->f1_ref.assign(f1, f1 + n_edge); h->f2_ref.assign(f2, f2 + n_edge);
    std::string terr = build_topology(n_real, n_face, n_edge, f1, f2, h->opt.reorder != 0,
                                      (h->gauss_seidel || h->tiny) ? h->opt.precond_colors : 0,
                                      (h->gauss_seidel || h->tiny) ? flow_hint : nullptr, h->world, h->topo,
                                      h->strips ? h->n_strips : 0, h->strip_cap);
    if (!terr.empty()) FAIL(CWR_EINVAL, terr);
    if (flow_hint) h->hint_done = true;
    const Topology& tp = h->topo;
    if (h->tma && (tp.W != 4 || tp.max_strip_nbr > 31)) { h->tma = false; h->opt.precond_sync = 3; }
    h->n = tp.n; h->F = tp.F; h->E = tp.E; h->G = tp.G; h->K = n_const; h->T = n_time;
    const int n = h->n, E = h->E, K = h->K, T = h->T;
    h->C = (h->opt.hydro_capacity <= 0 || h->opt.hydro_capacity > T) ? T : std::max(2, h->opt.hydro_capacity);
    const int kc = h->KC;
    h->max_grid = h->num_sms * 8;
    // persistent single-wave grids: SM count x resident CTAs per SM of the kernel that owns the grid
    {
        int occ_spmm = 4, occ_xrp = 3;
        KC_DISPATCH(h->KC, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_spmm, k_spmm<KC, VEC, MODE_AT, double>, kThreads, 0));
        KC_DISPATCH(h->KC, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_xrp, k_update_xrp<KC, VEC, double>, kThreads, 0));
        const int n_own = tp.part_ptr[h->rank + 1] - tp.part_ptr[h->rank];
        int occ_av = occ_spmm;
        KC_DISPATCH(h->KC, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ_av, k_spmm<KC, VEC, MODE_AV, double>, kThreads, 0));
        h->grid_at = grid_for(n_own, kThreads / kc, h->num_sms * std::max(1, occ_spmm));
        h->grid_spmm = grid_for(n_own, kThreads / kc, h->num_sms * std::max(1, occ_av));
        h->grid_xrp = grid_for(n_own, kThreads / kc, h->num_sms * std::max(1, occ_xrp));
        h->grid_sweep = grid_for(n_own, kThreads / h->SKC, h->num_sms * CWR_SPMM_MIN_BLOCKS);
    }
    if (h->tiny) {
        const size_t need = tiny_smem_bytes(n, tp.W);
        int max_optin = 0;
        cudaDeviceGetAttribute(&max_optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, device);
        if (need + kTinyStaticSmem > (size_t)max_optin) h->tiny = false;      // falls back to k_solve_small (Jacobi steps, any row order)
        else {
            h->tiny_rpt = (n + kTinyThreads - 1) / kTinyThreads;
            cudaError_t e = cudaSuccess;
            TINY_DISPATCH(e = cudaFuncSetAttribute(k_solve_tiny<RPT, W4>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)need));
            CK(e);
            CK(cudaFuncSetAttribute(k_solve_chip<8, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<8, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<12, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<12, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<14, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<14, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<8, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<8, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<12, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<12, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<14, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            CK(cudaFuncSetAttribute(k_solve_chip<14, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, max_optin - kTinyStaticSmem));
            h->max_optin_smem = max_optin;
            choose_chip(h);
        }
    }
    h->grid_rows = grid_for(tp.part_ptr[h->rank + 1] - tp.part_ptr[h->rank], kThreads / kc, h->max_grid);
    h->grid_edges = grid_for(E / h->world + 1, kThreads / kc, h->max_grid);
    h->grid_b = grid_for((int64_t)(tp.bcell.size() / h->world + 1) * K, kThreads, h->max_grid);

    // topology -> device
    CK(dalloc(h, &h->d_ell_col, tp.ell_col.size())); CK(dalloc(h, &h->d_ell_code, tp.ell_code.size()));
    CK(dalloc(h, &h->d_f1p, tp.f1p.size())); CK(dalloc(h, &h->d_f2p, tp.f2p.size()));
    CK(dalloc(h, &h->d_bcell, tp.bcell.size())); CK(dalloc(h, &h->d_bptr, tp.bptr.size())); CK(dalloc(h, &h->d_bedge, tp.bedge.size()));
    CK(dalloc(h, &h->d_eperm, (size_t)E)); CK(dalloc(h, &h->d_einv, (size_t)E));
    CK(dalloc(h, &h->d_new_of_old, (size_t)n)); CK(dalloc(h, &h->d_old_of_new, (size_t)n));
    CK(dalloc(h, &h->d_color_ptr, tp.color_ptr.size()));
    CK(dalloc(h, &h->d_send_mask, (size_t)n)); CK(dalloc(h, &h->d_send_rows, (size_t)n));
    if (h->strips) {
        CK(dalloc(h, &h->d_strip_cptr, tp.strip_cptr.size())); CK(dalloc(h, &h->d_strip_nptr, tp.strip_nptr.size()));
        CK(dalloc(h, &h->d_strip_flag, (size_t)h->n_strips * kFlagStride));
        CK(cudaMemsetAsync(h->d_strip_flag, 0, (size_t)h->n_strips * kFlagStride * sizeof(unsigned long long), h->stream));
        CK(dalloc(h, &h->d_strip_peers, tp.strip_peers.size()));
        if ((size_t)h->world * h->n_strips * kFlagStride * sizeof(unsigned long long) > kDdCtlBytes - kDdFlagOffset)
            FAIL(CWR_EINVAL, "too many strips for the flag mirrors of a domain decomposition");
    }
    {
        int rc = upload_topology(h);
        if (rc) return rc;
        std::vector<int32_t> a(f1, f1 + E), b(f2, f2 + E);
        CK(upload(h, &h->d_f1, a)); CK(upload(h, &h->d_f2, b));
        CK(cudaStreamSynchronize(h->stream));   // the vectors above die here
    }

    // hydro window, inputs, state, work vectors
    const size_t nK = (size_t)n * K;
    CK(dalloc(h, &h->d_adv, (size_t)h->C * E)); CK(dalloc(h, &h->d_cdiff, (size_t)h->C * E));
    CK(dalloc(h, &h->d_velg, (size_t)h->C * std::max(1, tp.E_g))); CK(dalloc(h, &h->d_vol, (size_t)h->C * n));
    CK(dalloc(h, &h->d_flowg, (size_t)h->C * std::max(1, tp.E_g)));
    CK(dalloc(h, &h->d_bc, (size_t)T * std::max(1, h->G) * K));
    CK(cudaMemsetAsync(h->d_bc, 0, (size_t)T * std::max(1, h->G) * K * sizeof(double), h->stream));
    h->n_state_slots = h->opt.keep_history ? T : 2;
    // Symmetric slab (same layout on every rank): DdCtl | p^ | s^ | tmp | state slots -- the vectors other
    // ranks gather from.  One allocation so that one CUDA IPC handle maps all of it into the peers.
    const bool need_precond_vectors = h->m_steps > 1 || h->small_path;
    const size_t vec_bytes = (nK * sizeof(double) + 255) & ~(size_t)255;
    h->slab_bytes = kDdCtlBytes + (need_precond_vectors ? 3 : 0) * vec_bytes + (size_t)h->n_state_slots * nK * sizeof(double);
    if (cudaMalloc((void**)&h->d_slab, h->slab_bytes) != cudaSuccess) {
        cudaGetLastError();
        FAIL(CWR_ENOMEM, "not enough device memory for the concentration history; set keep_history = 0");
    }
    h->allocs.push_back(h->d_slab);
    CK(cudaMemsetAsync(h->d_slab, 0, h->slab_bytes, h->stream));
    h->d_state = (double*)(h->d_slab + kDdCtlBytes + (need_precond_vectors ? 3 : 0) * vec_bytes);

    DeviceModel& M = h->M;
    M.n = n; M.K = K; M.E = E; M.E_int = tp.E_int; M.E_g = tp.E_g; M.G = h->G; M.nb = (int)tp.bcell.size();
    M.W = tp.W; M.ell_col = h->d_ell_col; M.ell_code = h->d_ell_code; M.f1p = h->d_f1p; M.f2p = h->d_f2p;
    M.bcell = h->d_bcell; M.bptr = h->d_bptr; M.bedge = h->d_bedge;
    M.rank = h->rank; M.world = h->world;
    M.send_mask = h->d_send_mask;
    M.dd = (DdCtl*)h->d_slab; M.sym_base = h->d_slab;
    for (int q = 0; q < kMaxRanks; ++q) M.peer_base[q] = nullptr;
    M.peer_base[h->rank] = h->d_slab;
    set_owned_ranges(h);
    CK(dalloc(h, &M.val, (size_t)n * tp.W)); CK(dalloc(h, &M.diag, (size_t)n)); CK(dalloc(h, &M.gdiag, (size_t)n));
    CK(cudaMemsetAsync(M.gdiag, 0, (size_t)n * sizeof(double), h->stream));
    double* ic = nullptr;
    CK(dalloc(h, &ic, nK)); CK(cudaMemsetAsync(ic, 0, nK * sizeof(double), h->stream));
    M.ic = ic;
    CK(dalloc(h, &M.b, nK)); CK(dalloc(h, &M.r, nK));
    CK(cudaMemsetAsync(M.b, 0, nK * sizeof(double), h->stream)); CK(cudaMemsetAsync(M.r, 0, nK * sizeof(double), h->stream));
    {   // the Krylov vectors (the defect-correction solver only needs them if it ever falls back: allocated either way,
        // 4 x 128 MB at 1M x 16 of 180 GB); all zeroed: t is multiplied by omega = 0 when a solve ends at a half step
        // before t = A s^ was ever formed, and no kernel may ever gather uninitialised rows
        double** vs[] = {&M.rhat, &M.p, &M.v, &M.tt};
        for (double** v : vs) { CK(dalloc(h, v, nK)); CK(cudaMemsetAsync(*v, 0, nK * sizeof(double), h->stream)); }
    }
    if (need_precond_vectors) {
        double* us;
        CK(dalloc(h, &us, nK));
        CK(cudaMemsetAsync(us, 0, nK * sizeof(double), h->stream));
        M.ph = h->d_slab + kDdCtlBytes; M.sh = h->d_slab + kDdCtlBytes + vec_bytes; M.tmp = h->d_slab + kDdCtlBytes + 2 * vec_bytes;
        M.us = us;
        if (h->sweep_f32 && (!h->small_path || h->tiny)) CK(dalloc(h, &M.valf, (size_t)n * tp.W));     // (on chip: k_solve_chip's fp32 sweeps)
    }
    if (h->small_path) {
        CK(dalloc(h, &M.xc, nK));
        CK(dalloc(h, &h->d_stats, 1));
        CK(cudaMemsetAsync(h->d_stats, 0, sizeof(SmallStats), h->stream));
        CK(cudaMallocHost((void**)&h->h_stats, sizeof(SmallStats)));
    }
    CK(dalloc(h, &M.partials, (size_t)h->max_grid * kMaxDots * K));
    CK(dalloc(h, &M.sc, (size_t)SC_ROWS * K));
    CK(dalloc(h, &M.colflags, (size_t)K)); CK(dalloc(h, &M.coliters, (size_t)K));
    CK(cudaMemsetAsync(M.colflags, 0, K * sizeof(int), h->stream));
    CK(cudaMemsetAsync(M.coliters, 0, K * sizeof(int), h->stream));
    CK(dalloc(h, &M.ctl, 1)); CK(cudaMemsetAsync(M.ctl, 0, sizeof(SolverCtl), h->stream));
    CK(dalloc(h, &h->d_sp, 1)); CK(cudaMemsetAsync(h->d_sp, 0, sizeof(StepParams), h->stream));
    M.sp = h->d_sp;
    M.want_flux = h->opt.mass_flux;
    if (M.want_flux) {
        CK(dalloc(h, &M.flux, (size_t)3 * E * K));
        CK(dalloc(h, &M.bsum, (size_t)3 * std::max(1, tp.E_g) * K));
        CK(cudaMemsetAsync(M.bsum, 0, (size_t)3 * std::max(1, tp.E_g) * K * sizeof(double), h->stream));
        CK(dalloc(h, &M.vsum, (size_t)3 * std::max(1, tp.E_g)));
        CK(cudaMemsetAsync(M.vsum, 0, (size_t)3 * std::max(1, tp.E_g) * sizeof(double), h->stream));
    }
    // what one cycle in the sweep precision can gain: measured on the 1M x 16 benchmark, fp32 cycles of 9 - 10 sweeps still
    // gain their full 0.2^S (3e5 / 10 planned three cycles of ~6 sweeps: 1.81 ms per step; 1e7 / 12 two of 9 - 10: 1.67)
    M.dc_smin = 2; M.dc_smax = h->sweep_f32 ? 12 : 24; M.dc_floor = h->sweep_f32 ? 1e7 : 1e12;
    if (h->dc_fixed) M.dc_smin = M.dc_smax = std::max(1, h->m_steps - 1);   // precond_steps given: every cycle does m - 1 sweeps
    M.sweep_f32 = h->sweep_f32 ? 1 : 0;
    M.us_from_producer = (h->dc && h->pipelined) ? 1 : 0;
    M.tol2 = h->opt.rtol * h->opt.rtol;
    M.diffusion_coefficient = D;
    M.max_iter = h->opt.max_iter;

    CK(cudaHostAlloc((void**)&h->h_mirror, sizeof(HostMirror), cudaHostAllocMapped));
    std::memset(h->h_mirror, 0, sizeof(HostMirror));
    CK(cudaHostGetDevicePointer((void**)&h->d_mirror, h->h_mirror, 0));
    h->h_ctl = &h->h_mirror->ctl; h->h_sc = h->h_mirror->sc; h->h_flags = h->h_mirror->flags;
    h->dt.assign(T, NAN);
    h->slot_time.assign(h->C, -1);
    h->initial_row.assign(K, std::vector<double>());
    h->inputs_set.assign(K, 0);
    h->real_overrides.resize(K);
    CK(cudaStreamSynchronize(h->stream));
    return CWR_OK;
}

int cwr_create(cwr_handle** out, int device, int n_real, int n_face, int n_edge, int n_time, int n_const,
               const int32_t* f1, const int32_t* f2, double D, const cwr_options* opt) {
    return cwr_create_with_hint(out, device, n_real, n_face, n_edge, n_time, n_const, f1, f2, D, opt, nullptr);
}

int cwr_create_with_hint(cwr_handle** out, int device, int n_real, int n_face, int n_edge, int n_time, int n_const,
                         const int32_t* f1, const int32_t* f2, double D, const cwr_options* opt, const float* flow_hint) {
    if (!out) return CWR_EINVAL;
    *out = nullptr;
    cwr_handle* h = new cwr_handle();
    int rc = create_impl(h, device, n_real, n_face, n_edge, n_time, n_const, f1, f2, D, opt, flow_hint);
    if (rc != CWR_OK) {
        g_create_error = h->err;
        cwr_destroy(h);
        return rc;
    }
    *out = h;
    return CWR_OK;
}

// ------------------------------------------------------------------------------------------------
// inputs
// ------------------------------------------------------------------------------------------------
static int check_slices(cwr_handle* h, int t0, int nt) {
    if (t0 < 0 || nt <= 0 || t0 + nt > h->T) FAIL(CWR_EINVAL, "time slice range outside [0, n_time)");
    if (nt > h->C) FAIL(CWR_EINVAL, "more slices than hydro_capacity in one call");
    return CWR_OK;
}

static int join_prefetch(cwr_handle* h, int slot = -1);

int cwr_set_hydro(cwr_handle* h, int t0, int nt, const float* adv, const double* cdiff, const float* vel,
                  const float* vol, const double* dt) {
    if (!h) return CWR_EINVAL;
    if (!adv || !cdiff || !vel || !vol || !dt) FAIL(CWR_EINVAL, "NULL array");
    int rc = check_slices(h, t0, nt);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    rc = align_colours_with_flow(h, adv, nt);
    if (rc) return rc;
    rc = join_prefetch(h);
    if (rc) return rc;
    const int n = h->n, E = h->E, F = h->F, Eg = h->topo.E_g, Ei = h->topo.E_int;
    // staging: adv f32 (E) | vel f32 (E) | vol f32 (F) | cdiff f64 (E)
    const size_t off_vel = (size_t)E * 4, off_vol = off_vel + (size_t)E * 4, off_cd = (off_vol + (size_t)F * 4 + 7) & ~(size_t)7;
    rc = ensure_stage(h, off_cd + (size_t)E * 8);
    if (rc) return rc;
    char* st = (char*)h->d_stage;
    const int g = grid_for(E, kThreads, h->max_grid);
    for (int s = 0; s < nt; ++s) {
        const int t = t0 + s, slot = t % h->C;
        CK(cudaMemcpyAsync(st, adv + (size_t)s * E, (size_t)E * 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(st + off_vel, vel + (size_t)s * E, (size_t)E * 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(st + off_vol, vol + (size_t)s * F, (size_t)F * 4, cudaMemcpyHostToDevice, h->stream));
        CK(cudaMemcpyAsync(st + off_cd, cdiff + (size_t)s * E, (size_t)E * 8, cudaMemcpyHostToDevice, h->stream));
        k_gather<float><<<g, kThreads, 0, h->stream>>>(h->d_adv + (size_t)slot * E, (const float*)st, h->d_eperm, E);
        k_gather<double><<<g, kThreads, 0, h->stream>>>(h->d_cdiff + (size_t)slot * E, (const double*)(st + off_cd), h->d_eperm, E);
        if (Eg > 0)
            k_gather<float><<<grid_for(Eg, kThreads, h->max_grid), kThreads, 0, h->stream>>>(
                h->d_velg + (size_t)slot * Eg, (const float*)(st + off_vel), h->d_eperm + Ei, Eg);
        if (Eg > 0)     // (the raw face flow is not given on this path: advection_coeff = face_flow * sign(|velocity|) stands in)
            k_gather<float><<<grid_for(Eg, kThreads, h->max_grid), kThreads, 0, h->stream>>>(
                h->d_flowg + (size_t)slot * Eg, (const float*)st, h->d_eperm + Ei, Eg);
        k_gather<float><<<grid_for(n, kThreads, h->max_grid), kThreads, 0, h->stream>>>(
            h->d_vol + (size_t)slot * n, (const float*)(st + off_vol), h->d_old_of_new, n);
        h->launches += 4;
        h->dt[t] = dt[s];
        h->slot_time[slot] = t;
    }
    CK(cudaGetLastError());
    return CWR_OK;
}

int cwr_set_flow_hint(cwr_handle* h, const float* face_flow) {
    if (!h) return CWR_EINVAL;
    if (!face_flow) FAIL(CWR_EINVAL, "NULL array");
    for (int t : h->slot_time) if (t >= 0) FAIL(CWR_EINVAL, "cwr_set_flow_hint must come before the first hydrodynamic slice");
    for (uint8_t s : h->inputs_set) if (s) FAIL(CWR_EINVAL, "cwr_set_flow_hint must come before cwr_set_inputs");
    CK(cudaSetDevice(h->device));
    return align_colours_with_flow(h, face_flow, 1);
}

int cwr_set_geometry(cwr_handle* h, const double* face_x, const double* face_y) {
    if (!h) return CWR_EINVAL;
    if (!face_x || !face_y) FAIL(CWR_EINVAL, "NULL array");
    CK(cudaSetDevice(h->device));
    int rc = ensure_stage(h, (size_t)2 * h->F * 8);
    if (rc) return rc;
    double* fx = (double*)h->d_stage; double* fy = fx + h->F;
    CK(cudaMemcpyAsync(fx, face_x, (size_t)h->F * 8, cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(fy, face_y, (size_t)h->F * 8, cudaMemcpyHostToDevice, h->stream));
    if (!h->d_dist) CK(dalloc(h, &h->d_dist, (size_t)h->E));
    k_dist<<<grid_for(h->E, kThreads, h->max_grid), kThreads, 0, h->stream>>>(h->d_dist, fx, fy, h->d_f1, h->d_f2, h->E);
    h->launches += 1;
    CK(cudaGetLastError());
    h->have_geometry = true;
    return CWR_OK;
}

// slices [t0, t0+nt) of the raw arrays -> device order + derived coefficients, on `stream` through staging buffer `st`
static int upload_raw(cwr_handle* h, cudaStream_t stream, char* st, int t0, int nt, const float* face_flow,
                      const float* edge_velocity, const float* volume, const double* dt) {
    const int n = h->n, E = h->E, F = h->F, Eg = h->topo.E_g, Ei = h->topo.E_int;
    const size_t off_vel = (size_t)E * 4, off_vol = off_vel + (size_t)E * 4;
    for (int s = 0; s < nt; ++s) {
        const int t = t0 + s, slot = t % h->C;
        CK(cudaMemcpyAsync(st, face_flow + (size_t)s * E, (size_t)E * 4, cudaMemcpyHostToDevice, stream));
        CK(cudaMemcpyAsync(st + off_vel, edge_velocity + (size_t)s * E, (size_t)E * 4, cudaMemcpyHostToDevice, stream));
        CK(cudaMemcpyAsync(st + off_vol, volume + (size_t)s * F, (size_t)F * 4, cudaMemcpyHostToDevice, stream));
        k_derive<<<grid_for(E, kThreads, h->max_grid), kThreads, 0, stream>>>(
            h->d_adv + (size_t)slot * E, h->d_cdiff + (size_t)slot * E, h->d_velg + (size_t)slot * std::max(1, Eg),
            h->d_flowg + (size_t)slot * std::max(1, Eg),
            (const float*)st, (const float*)(st + off_vel), h->d_dist, h->d_eperm, E, Ei, (float)h->M.diffusion_coefficient);
        k_gather<float><<<grid_for(n, kThreads, h->max_grid), kThreads, 0, stream>>>(
            h->d_vol + (size_t)slot * n, (const float*)(st + off_vol), h->d_old_of_new, n);
        h->launches += 2;
        h->dt[t] = dt[s];
        h->slot_time[slot] = t;
    }
    CK(cudaGetLastError());
    return CWR_OK;
}

// the compute stream must see a prefetched slice before it reads the hydro window again
// (slot < 0: every slot)
static int join_prefetch(cwr_handle* h, int slot) {
    for (int s = 0; s < (int)h->up_pending.size(); ++s) {
        if ((slot >= 0 && s != slot) || !h->up_pending[s]) continue;
        CK(cudaStreamWaitEvent(h->stream, h->up_done[s], 0));
        h->up_pending[s] = 0;
    }
    return CWR_OK;
}

int cwr_set_hydro_raw(cwr_handle* h, int t0, int nt, const float* face_flow, const float* edge_velocity,
                      const float* volume, const double* dt) {
    if (!h) return CWR_EINVAL;
    if (!face_flow || !edge_velocity || !volume || !dt) FAIL(CWR_EINVAL, "NULL array");
    if (!h->have_geometry) FAIL(CWR_EINVAL, "cwr_set_geometry must be called before cwr_set_hydro_raw");
    int rc = check_slices(h, t0, nt);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    rc = align_colours_with_flow(h, face_flow, nt);
    if (rc) return rc;
    rc = join_prefetch(h);
    if (rc) return rc;
    rc = ensure_stage(h, (size_t)h->E * 8 + (size_t)h->F * 4);
    if (rc) return rc;
    return upload_raw(h, h->stream, (char*)h->d_stage, t0, nt, face_flow, edge_velocity, volume, dt);
}

int cwr_prefetch_hydro_raw(cwr_handle* h, int t0, int nt, const float* face_flow, const float* edge_velocity,
                           const float* volume, const double* dt) {
    if (!h) return CWR_EINVAL;
    if (!face_flow || !edge_velocity || !volume || !dt) FAIL(CWR_EINVAL, "NULL array");
    if (!h->have_geometry) FAIL(CWR_EINVAL, "cwr_set_geometry must be called before cwr_prefetch_hydro_raw");
    int rc = check_slices(h, t0, nt);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    if (!h->up_stream) {
        CK(cudaStreamCreateWithFlags(&h->up_stream, cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&h->compute_mark, cudaEventDisableTiming));
        h->up_done.assign(h->C, nullptr); h->up_pending.assign(h->C, 0);
        for (int sl = 0; sl < h->C; ++sl) CK(cudaEventCreateWithFlags(&h->up_done[sl], cudaEventDisableTiming));
    }
    const size_t need = (size_t)h->E * 8 + (size_t)h->F * 4;
    if (need > h->stage_up_bytes) {
        if (h->d_stage_up) { CK(cudaStreamSynchronize(h->up_stream)); CK(cudaFree(h->d_stage_up)); h->d_stage_up = nullptr; }
        CK(cudaMalloc(&h->d_stage_up, need));
        h->stage_up_bytes = need;
    }
    // the slots being overwritten may still be read by work already queued on the compute stream
    CK(cudaEventRecord(h->compute_mark, h->stream));
    CK(cudaStreamWaitEvent(h->up_stream, h->compute_mark, 0));
    for (int s = 0; s < nt; ++s) {      // one event per slice: a step only waits for the two slices it reads
        rc = upload_raw(h, h->up_stream, (char*)h->d_stage_up, t0 + s, 1, face_flow + (size_t)s * h->E, edge_velocity + (size_t)s * h->E,
                        volume + (size_t)s * h->F, dt + s);
        if (rc) return rc;
        const int slot = (t0 + s) % h->C;
        CK(cudaEventRecord(h->up_done[slot], h->up_stream));
        h->up_pending[slot] = 1;
    }
    return CWR_OK;
}

int cwr_set_inputs(cwr_handle* h, int k, const double* input) {
    if (!h) return CWR_EINVAL;
    if (!input) FAIL(CWR_EINVAL, "NULL array");
    if (k < 0 || k >= h->K) FAIL(CWR_EINVAL, "constituent index out of range");
    CK(cudaSetDevice(h->device));
    const int n = h->n, F = h->F, G = h->G, T = h->T, K = h->K;
    // host: initial row (constituents.py:94-98) and BC block packed (T,G)
    std::vector<double>& row0 = h->initial_row[k];
    row0.assign(F, 0.0);
    std::copy(input, input + n, row0.begin());
    std::vector<double> pack((size_t)T * std::max(1, G));
    for (int t = 0; t < T; ++t) std::copy(input + (size_t)t * F + n, input + (size_t)t * F + F, pack.begin() + (size_t)t * G);
    // real-cell entries at t >= 1 that are non-zero override c~ (linalg.py:199-200); rare
    auto& ov = h->real_overrides[k];
    ov.clear();
    for (int t = 1; t < T; ++t) {
        const double* r = input + (size_t)t * F;
        for (int i = 0; i < n; ++i)
            if (r[i] != 0.0) ov[t].emplace_back(h->topo.new_of_old[i], r[i]);
    }
    int rc = ensure_stage(h, std::max(pack.size(), (size_t)n) * 8 + (size_t)n * 8);
    if (rc) return rc;
    double* st = (double*)h->d_stage;
    CK(cudaMemcpyAsync(st, input, (size_t)n * 8, cudaMemcpyHostToDevice, h->stream));
    const int g = grid_for(n, kThreads, h->max_grid);
    k_scatter_column<<<g, kThreads, 0, h->stream>>>((double*)h->M.ic, st, h->d_old_of_new, n, K, k);
    k_scatter_column<<<g, kThreads, 0, h->stream>>>(h->d_state, st, h->d_old_of_new, n, K, k);   // c[0]
    h->launches += 2;
    CK(cudaStreamSynchronize(h->stream));
    if (G > 0) {
        CK(cudaMemcpyAsync(st, pack.data(), pack.size() * 8, cudaMemcpyHostToDevice, h->stream));
        // input layout seen by the kernel: (T, G) with "F" = G and n = 0
        k_scatter_bc<<<grid_for((int64_t)T * G, kThreads, h->max_grid), kThreads, 0, h->stream>>>(h->d_bc, st, T, G, 0, G, K, k);
        h->launches += 1;
        CK(cudaStreamSynchronize(h->stream));
    }
    CK(cudaGetLastError());
    h->inputs_set[k] = 1;
    return CWR_OK;
}

static inline double* state_slot(cwr_handle* h, int t) {
    const int s = h->opt.keep_history ? t : (t & 1);
    return h->d_state + (size_t)s * h->n * h->K;
}

static int state_available(cwr_handle* h, int t) {
    if (t < 0 || t >= h->T) FAIL(CWR_EINVAL, "time index out of range");
    if (t > h->computed_upto) FAIL(CWR_EINVAL, "state at this time index has not been computed yet");
    if (!h->opt.keep_history && t < h->computed_upto - 1) FAIL(CWR_EINVAL, "state no longer on the device (keep_history = 0)");
    return CWR_OK;
}

int cwr_set_state(cwr_handle* h, int k, int t, const double* c) {
    if (!h) return CWR_EINVAL;
    if (!c) FAIL(CWR_EINVAL, "NULL array");
    if (k < 0 || k >= h->K) FAIL(CWR_EINVAL, "constituent index out of range");
    int rc = state_available(h, t);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    rc = ensure_stage(h, (size_t)h->n * 8);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h->d_stage, c, (size_t)h->n * 8, cudaMemcpyHostToDevice, h->stream));
    k_scatter_column<<<grid_for(h->n, kThreads, h->max_grid), kThreads, 0, h->stream>>>(
        state_slot(h, t), (const double*)h->d_stage, h->d_old_of_new, h->n, h->K, k);
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return CWR_OK;
}

int cwr_set_state_all(cwr_handle* h, int t, const double* c, const uint8_t* mask) {
    if (!h) return CWR_EINVAL;
    if (!c) FAIL(CWR_EINVAL, "NULL array");
    int rc = state_available(h, t);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    const size_t nK = (size_t)h->n * h->K;
    rc = ensure_stage(h, nK * 8 + 256);
    if (rc) return rc;
    uint8_t* dmask = nullptr;
    CK(cudaMemcpyAsync(h->d_stage, c, nK * 8, cudaMemcpyHostToDevice, h->stream));
    if (mask) {
        dmask = (uint8_t*)h->d_stage + nK * 8;
        CK(cudaMemcpyAsync(dmask, mask, h->K, cudaMemcpyHostToDevice, h->stream));
    }
    k_scatter_all<<<grid_for((int64_t)nK, kThreads, h->max_grid), kThreads, 0, h->stream>>>(
        state_slot(h, t), (const double*)h->d_stage, dmask, h->d_new_of_old, h->n, h->K);
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cudaStreamSynchronize(h->stream));
    return CWR_OK;
}

// ------------------------------------------------------------------------------------------------
// one step
// ------------------------------------------------------------------------------------------------
static int poll(cwr_handle* h, int with_columns = 0) {
    k_mirror<<<1, 128, 0, h->stream>>>(h->M.ctl, h->M.sc, h->M.colflags, h->K, h->d_mirror, with_columns);
    CK(cudaStreamSynchronize(h->stream));
    return CWR_OK;
}

// z = M^-1 u with m - 1 sweeps, result in `dst` (sweep type); returns u itself when m == 1.
//   Jacobi:        z_1 = u + N u, z_{j+1} = u + N z_j  (N = I - D^-1 A)  =>  z = (I + N + ... + N^(m-1)) u
//   Gauss-Seidel:  the same first step, then m - 2 in-place multicolour sweeps (one launch per colour)
static const void* precondition(cwr_handle* h, const double* u, void* dst, void* other, bool planned = false) {
    const int J = h->m_steps - 1;
    if (J <= 0) return u;
    DeviceModel& M = h->M;
    if (h->gauss_seidel) {
        mark(h, CWR_FAM_PRECOND);
        int sweeps = planned ? 0 : J;                 // 0: the count the defect-correction solver planned on the device
        unsigned long long seq = ++h->gs_seq;
        void* args[] = {(void*)&M, (void*)&u, (void*)&dst, (void*)&sweeps, (void*)&seq};
        cudaError_t e = cudaSuccess;
        if (h->pipelined) {
            if (!M.us_from_producer) {        // BiCGSTAB: u is one of its fp64 vectors
                if (h->sweep_f32) k_to_sweep_type<float><<<h->grid_rows, kThreads, 0, h->stream>>>(M, u, (float*)M.us);
                else k_to_sweep_type<double><<<h->grid_rows, kThreads, 0, h->stream>>>(M, u, (double*)M.us);
                h->launches += 1;
            }
            void* args3[] = {(void*)&M, (void*)&dst, (void*)&sweeps, (void*)&seq};
            if (h->tma && h->gs_debug) {          // development: timing experiments (see k_gs_tma)
                int packed = sweeps | (h->gs_debug << 16);
                void* argsd[] = {(void*)&M, (void*)&dst, (void*)&packed};
                e = cudaLaunchCooperativeKernel((const void*)k_gs_tma<true>, dim3(h->grid_gs), dim3(kGsThreads), argsd, kTmaSmemBytes, h->stream);
            } else if (h->tma) e = cudaLaunchCooperativeKernel((const void*)k_gs_tma<false>, dim3(h->grid_gs), dim3(kGsThreads), args3, kTmaSmemBytes, h->stream);
            else SWEEP_DISPATCH(e = (gs3_launch<ST, SKC, SVEC>(h->grid_gs, args3, h->stream)));
        } else
        if (h->strips) { SWEEP_DISPATCH(e = cudaLaunchCooperativeKernel((const void*)k_precond_gs<ST, SKC, SVEC, true>, dim3(h->grid_gs), dim3(kGsThreads), args, kGsSmemBytes, h->stream)); }
        else { SWEEP_DISPATCH(e = cudaLaunchCooperativeKernel((const void*)k_precond_gs<ST, SKC, SVEC, false>, dim3(h->grid_gs), dim3(kGsThreads), args, kGsSmemBytes, h->stream)); }
        if (e != cudaSuccess) h->err = std::string("k_precond_gs: ") + cudaGetErrorString(e);
        h->launches += 1;
        return dst;
    }
    const void* z = nullptr;
    for (int j = 1; j <= J; ++j) {
        void* out = ((J - j) % 2 == 0) ? dst : other;      // the last step always lands in dst
        mark(h, CWR_FAM_PRECOND);
        if (j == 1) { SWEEP_DISPATCH((k_sweep<ST, SKC, SVEC, true><<<h->grid_sweep, kThreads, 0, h->stream>>>(M, u, nullptr, (ST*)out, M.row_lo, M.row_hi))); }
        else { SWEEP_DISPATCH((k_sweep<ST, SKC, SVEC, false><<<h->grid_sweep, kThreads, 0, h->stream>>>(M, nullptr, (const ST*)z, (ST*)out, M.row_lo, M.row_hi))); }
        h->launches += 1;
        if (h->world > 1) { if (h->sweep_f32) halo_push(h, (float*)out); else halo_push(h, (double*)out); }
        z = out;
    }
    return z;
}

static int launch_iteration(cwr_handle* h) {
    const int g = h->grid_rows;
    DeviceModel& M = h->M;
    const void* ph = precondition(h, M.p, M.ph, M.tmp);
    mark(h, CWR_FAM_SPMM_V);
    PT_DISPATCH((k_spmm<KC, VEC, MODE_AV, PT><<<h->grid_spmm, kThreads, 0, h->stream>>>(M, (const PT*)ph, nullptr)));
    mark(h, CWR_FAM_UPDATE_S);
    KC_DISPATCH(h->KC, (k_update_s<KC, VEC><<<g, kThreads, 0, h->stream>>>(M)));
    const void* sh = precondition(h, M.r, M.sh, M.tmp);
    mark(h, CWR_FAM_SPMM_T);
    PT_DISPATCH((k_spmm<KC, VEC, MODE_AT, PT><<<h->grid_at, kThreads, 0, h->stream>>>(M, (const PT*)sh, nullptr)));
    mark(h, CWR_FAM_UPDATE_XRP);
    PT_DISPATCH((k_update_xrp<KC, VEC, PT><<<h->grid_xrp, kThreads, 0, h->stream>>>(M, (const PT*)ph, (const PT*)sh)));
    h->launches += 4;
    return CWR_OK;
}

static int solve(cwr_handle* h, cwr_step_info* info) {
    DeviceModel& M = h->M;
    int restarts = 0;
    int total_iter = 0;
    for (;;) {
        mark(h, CWR_FAM_SPMM_INIT);
        KC_DISPATCH(h->KC, (k_spmm<KC, VEC, MODE_INIT, double><<<h->grid_spmm, kThreads, 0, h->stream>>>(M, nullptr, nullptr)));
        h->launches += 1;
        mark(h, -1);
        // Launch-ahead: the previous solve's iteration count predicts this one, so that many iterations
        // (minus one) are queued before the first convergence poll; every kernel of an iteration returns
        // at once when the device-side all_done flag is already set, so over-launching is harmless.
        int ahead = restarts == 0 ? std::max(0, h->last_iters - 1) : 0;
        int rc = CWR_OK;
        if (ahead == 0) { rc = poll(h); if (rc) return rc; } else h->h_ctl->all_done = 0;
        while (!h->h_ctl->all_done) {
            const int burst = ahead > 0 ? ahead : h->opt.check_every;
            ahead = 0;
            for (int i = 0; i < burst; ++i) launch_iteration(h);
            mark(h, -1);
            rc = poll(h);
            if (rc) return rc;
        }
        h->last_iters = h->h_ctl->iter;
        total_iter += h->h_ctl->iter;
        const bool breakdown = (h->h_ctl->flags_or & FL_BREAKDOWN) != 0;
        if (breakdown && restarts < 3 && !h->h_ctl->hit_max_iter) {
            // restart from the current iterate: new shadow residual (standard cure for rho ~ 0)
            ++restarts;
            CK(cudaMemsetAsync(&M.ctl->all_done, 0, 2 * sizeof(int), h->stream));   // all_done, iter
            // domain decomposition: the new residual gathers the neighbours' rows of the CURRENT iterate
            { int rch = halo_push(h, h->cur_x); if (rch) return rch; }
            continue;
        }
        break;
    }
    CK(cudaGetLastError());
    { int rcp = poll(h, 1); if (rcp) return rcp; }
    h->iterations += total_iter;
    int status = CWR_OK;
    double worst = 0.0;
    for (int k = 0; k < h->K; ++k) {
        const double bb = h->h_sc[SC_BNORM2 * h->K + k], rr = h->h_sc[SC_RNORM2 * h->K + k];
        const double rel = bb > 0 ? std::sqrt(rr / bb) : (rr > 0 ? INFINITY : 0.0);
        if (rel == rel) worst = std::max(worst, rel);
        const int f = h->h_flags[k];
        if (f & FL_NAN) status = CWR_ENAN;
        else if ((f & FL_BREAKDOWN) && !(f & FL_CONVERGED) && status == CWR_OK) status = CWR_EBREAKDOWN;
        else if (!(f & FL_CONVERGED) && status == CWR_OK) status = CWR_ENOTCONVERGED;
    }
    if (h->h_ctl->singular) status = CWR_ESINGULAR;
    if (h->h_ctl->barrier_timeout) { h->err = "a grid barrier timed out"; return CWR_ECUDA; }
    if (h->world > 1) {
        int dd_timeout = 0;
        CK(cudaMemcpyAsync(&dd_timeout, &h->M.dd->timeout, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (dd_timeout) { h->err = "a peer rank did not answer (halo barrier / dot-product exchange timed out)"; return CWR_ECUDA; }
    }
    if (info) { info->iterations = total_iter; info->restarts = restarts; info->status = status; info->max_relres = worst; }
    return status;
}

// Defect correction with the preconditioner sweeps as the solver (options.solver = 2):
//   r = b - A x0;  repeat { z = M^-1 r (fp32 Gauss-Seidel sweeps from 0);  x += z;  r -= A z }  until ||r|| <= rtol ||b||
// Gauss-Seidel sweeps on A z = r from z = 0 followed by x += z ARE Gauss-Seidel sweeps on A x = b: the cycle only
// exists to carry the residual and the iterate in fp64 around sweeps that run in fp32.  On the upwind M-matrices of
// this problem the flow-aligned sweeps contract the error by ~0.2 each, Krylov acceleration adds nothing, and the
// solve needs neither the Krylov vectors' traffic nor their dot products: one reduction per cycle, for the
// convergence test.  The sweeps per cycle are planned on the device (dc_plan); the cycles of the previous solve are
// queued before the first poll, every kernel of a cycle returns at once when all_done is set.
// Returns 1 when the sweeps stagnate or diverge (the matrix is not what the sweeps assume): the caller restores
// x0 and solves with BiCGSTAB.
static int solve_dc(cwr_handle* h, cwr_step_info* info, bool* fell_back) {
    DeviceModel& M = h->M;
    *fell_back = false;
    mark(h, CWR_FAM_SPMM_INIT);
    KC_DISPATCH(h->KC, (k_spmm<KC, VEC, MODE_INIT_DC, double><<<h->grid_spmm, kThreads, 0, h->stream>>>(M, nullptr, nullptr)));
    h->launches += 1;
    mark(h, -1);
    int ahead = std::max(1, h->last_cycles);
    h->h_ctl->all_done = 0;
    int rc = CWR_OK;
    int launched = 0;
    while (!h->h_ctl->all_done) {
        const int burst = ahead > 0 ? ahead : h->opt.check_every;
        ahead = 0;
        for (int i = 0; i < burst; ++i) {
            const void* z = precondition(h, M.r, M.ph, M.tmp, true);
            mark(h, CWR_FAM_DC_UPDATE);
            PT_DISPATCH((k_spmm<KC, VEC, MODE_DC, PT><<<h->grid_spmm, kThreads, 0, h->stream>>>(M, (const PT*)z, nullptr)));
            h->launches += 1;
            ++launched;
        }
        mark(h, -1);
        rc = poll(h);
        if (rc) return rc;
        if (launched > h->opt.max_iter + 8) break;       // (the device sets hit_max_iter long before)
    }
    CK(cudaGetLastError());
    h->last_cycles = h->h_ctl->iter;
    h->sweeps_total += h->h_ctl->sweeps_done;
    if (h->h_ctl->barrier_timeout) { h->err = "a sweep-kernel barrier timed out"; return CWR_ECUDA; }
    if (h->h_ctl->dc_fail) { *fell_back = true; return CWR_OK; }
    if (h->h_ctl->flags_or & FL_PENDING) {          // NaN right-hand sides / b == 0: fill those columns
        k_fix_columns<<<grid_for((int64_t)(M.row_hi - M.row_lo) * h->K, kThreads, h->max_grid), kThreads, 0, h->stream>>>(M);
        k_fix_flags<<<1, 128, 0, h->stream>>>(M);
        h->launches += 2;
    }
    { int rcp = poll(h, 1); if (rcp) return rcp; }
    h->iterations += h->h_ctl->iter;
    int status = CWR_OK;
    double worst = 0.0;
    for (int k = 0; k < h->K; ++k) {
        const double bb = h->h_sc[SC_BNORM2 * h->K + k], rr = h->h_sc[SC_RNORM2 * h->K + k];
        const double rel = bb > 0 ? std::sqrt(rr / bb) : (rr > 0 ? INFINITY : 0.0);
        if (rel == rel) worst = std::max(worst, rel);
        const int f = h->h_flags[k];
        if (f & FL_NAN) status = CWR_ENAN;
        else if (!(f & FL_CONVERGED) && status == CWR_OK) status = CWR_ENOTCONVERGED;
    }
    if (h->h_ctl->singular) status = CWR_ESINGULAR;
    if (h->world > 1) {
        int dd_timeout = 0;
        CK(cudaMemcpyAsync(&dd_timeout, &h->M.dd->timeout, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
        if (dd_timeout) { h->err = "a peer rank did not answer (halo barrier / dot-product exchange timed out)"; return CWR_ECUDA; }
    }
    if (info) { info->iterations = h->h_ctl->iter; info->restarts = 0; info->status = status; info->max_relres = worst; info->sweeps = h->h_ctl->sweeps_done; }
    return status;
}

// Small-mesh path: the whole solve of every column is one launch; convergence is decided on the
// device.  Inside cwr_run nothing is read back per step (statistics accumulate in d_stats).
static int read_small_stats(cwr_handle* h, cwr_step_info* info) {
    CK(cudaMemcpyAsync(h->h_stats, h->d_stats, sizeof(SmallStats), cudaMemcpyDeviceToHost, h->stream));
    { int rcp = poll(h); if (rcp) return rcp; }
    const SmallStats& s = *h->h_stats;
    double rel2;
    std::memcpy(&rel2, &s.max_relres2_bits, sizeof rel2);
    int status = CWR_OK;
    if (s.flags_or & FL_NAN) status = CWR_ENAN;
    else if (s.flags_or & FL_BREAKDOWN) status = CWR_EBREAKDOWN;
    else if (s.not_converged > 0) status = CWR_ENOTCONVERGED;
    if (h->h_ctl->singular) status = CWR_ESINGULAR;
    if (info) { info->iterations = s.max_iterations; info->restarts = s.restarts; info->status = status; info->max_relres = std::sqrt(rel2); }
    return status;
}

static int solve_small(cwr_handle* h, cwr_step_info* info) {
    if (!h->in_run) CK(cudaMemsetAsync(h->d_stats, 0, sizeof(SmallStats), h->stream));
    mark(h, CWR_FAM_SOLVE_SMALL);
    if (h->tiny && h->chip_ns > 0) {
        const size_t sm = chip_smem_bytes(h->n, h->chip_ns);
        const int sweeps = h->m_steps - 1;
#define CHIP_LAUNCH(NS) do { \
            const bool full = h->topo.n_colors == NS; \
            if (h->sweep_f32 && full) CK(launch_chain(h, k_solve_chip<NS, true, true>, h->K, kChipThreads, sm, h->M, sweeps, h->d_stats)); \
            else if (h->sweep_f32) CK(launch_chain(h, k_solve_chip<NS, true, false>, h->K, kChipThreads, sm, h->M, sweeps, h->d_stats)); \
            else if (full) CK(launch_chain(h, k_solve_chip<NS, false, true>, h->K, kChipThreads, sm, h->M, sweeps, h->d_stats)); \
            else CK(launch_chain(h, k_solve_chip<NS, false, false>, h->K, kChipThreads, sm, h->M, sweeps, h->d_stats)); } while (0)
        if (h->chip_ns == 8) CHIP_LAUNCH(8);
        else if (h->chip_ns == 12) CHIP_LAUNCH(12);
        else CHIP_LAUNCH(14);
#undef CHIP_LAUNCH
    } else if (h->tiny) {
        const size_t sm = tiny_smem_bytes(h->n, h->topo.W);
        const int sweeps = h->m_steps - 1;
        TINY_DISPATCH((launch_chain(h, k_solve_tiny<RPT, W4>, h->K, kTinyThreads, sm, h->M, sweeps, h->d_stats)));
    } else
    CK(launch_chain(h, k_solve_small, h->K, kSmallThreads, 0, h->M, h->m_steps, h->d_stats));
    h->launches += 1;
    CK(cudaGetLastError());
    if (h->in_run) {
        if (info) { info->iterations = 0; info->restarts = 0; info->status = CWR_OK; info->max_relres = 0.0; }
        return CWR_OK;
    }
    int status = read_small_stats(h, info);
    if (status != CWR_ECUDA) h->iterations += (int64_t)(h->h_stats->sum_iterations / (unsigned long long)h->K);
    return status;
}

static int find_slot(cwr_handle* h, int t) {
    const int s = t % h->C;
    return h->slot_time[s] == t ? s : -1;
}

// sparse real-cell entries of input_array[t] (rare): one upload + one kernel for all constituents
static int patch_real_cells(cwr_handle* h, int t, int before_solve) {
    DeviceModel& M = h->M;
    h->ov_idx.clear(); h->ov_val.clear();
    for (int k = 0; k < h->K; ++k) {
        auto it = h->real_overrides[k].find(t);
        if (it == h->real_overrides[k].end()) continue;
        for (auto& cv : it->second)
            if (cv.first >= M.row_lo && cv.first < M.row_hi) {      // (another rank's rows are that rank's business)
                h->ov_idx.push_back((long long)cv.first * h->K + k);
                h->ov_val.push_back(cv.second);
            }
    }
    const size_t cnt = h->ov_idx.size();
    if (cnt == 0) return CWR_OK;
    if (cnt > h->ov_cap) {
        CK(cudaStreamSynchronize(h->stream));
        if (h->d_ov_idx) CK(cudaFree(h->d_ov_idx));
        if (h->d_ov_val) CK(cudaFree(h->d_ov_val));
        h->d_ov_idx = nullptr; h->d_ov_val = nullptr;
        h->ov_cap = cnt + cnt / 2 + 64;
        CK(cudaMalloc((void**)&h->d_ov_idx, h->ov_cap * sizeof(long long)));
        CK(cudaMalloc((void**)&h->d_ov_val, h->ov_cap * sizeof(double)));
    }
    // pageable sources: the copies have left the host vectors when the calls return
    CK(cudaMemcpyAsync(h->d_ov_idx, h->ov_idx.data(), cnt * sizeof(long long), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_ov_val, h->ov_val.data(), cnt * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(launch_chain(h, k_patch_rows, grid_for((int64_t)cnt, kThreads, 64), kThreads, 0, M, (const long long*)h->d_ov_idx, (const double*)h->d_ov_val, (int)cnt, before_solve));
    h->launches += 1;
    return CWR_OK;
}

// b and the warm start x0 = c~ of step t (after the LHS: b is row-scaled by the diagonal), reacted when kinetics is set,
// then x0's boundary rows to the ranks that gather them.  accumulate = 0 (the defect-correction fallback forms the same
// right-hand side again): the step's reaction mass is not added a second time.
static int build_rhs(cwr_handle* h, int t, int accumulate) {
    DeviceModel& M = h->M;
    mark(h, CWR_FAM_RHS);
    KC_DISPATCH(h->KC, (launch_chain(h, k_rhs<KC, VEC>, h->grid_rows, kThreads, 0, M)));
    h->launches += 1;
    int rc = patch_real_cells(h, t, 1);
    if (rc) return rc;
    if (h->kin_on) {
        // one CTA per tile of the rows this rank owns now (the ordering, and with it the row range, may still be rebuilt
        // after cwr_set_kinetics), at most the resident grid; the same rows give the same grid, hence the same sums
        const int R = react_tile_rows(h->K);
        const int grid = grid_for((M.row_hi - M.row_lo + R - 1) / R, 1, h->kin_grid_max);
        auto* fn = h->kin_forced ? (h->kin_depth ? k_react<true, true, true> : h->kin_facs ? k_react<true, false, true> : k_react<false, false, true>)
                                 : (h->kin_depth ? k_react<true, true> : h->kin_facs ? k_react<true> : k_react<false>);
        const int* fptr = h->kin_depth && !h->kin_facs ? h->d_kin_fptr0 : h->d_kin_fptr;
        const size_t smem = react_smem_bytes(h->K) + react_src_smem_bytes(h->kin_srcs, h->kin_temp_k) +
                            (h->kin_forced ? react_force_smem_bytes(h->kin_srcs) : 0);
        CK(launch_chain(h, fn, grid, kThreads, smem, M,
                        (const KinStep*)h->d_kin_steps, h->kin_steps, (const KinYield*)h->d_kin_yields, h->kin_temp_k, h->kin_temp_c,
                        (const KinSrc*)h->d_kin_srcs, h->kin_srcs, h->kin_src_o2, (const KinFac*)h->d_kin_facs,
                        fptr, h->d_kin_partials, h->d_kin_state, accumulate, (const double*)h->d_kin_area,
                        (const int*)h->d_kin_dflag, h->kin_min_depth));
        h->launches += 1;
    }
    if (M.b_hi - M.b_lo > 0) {
        CK(launch_chain(h, k_boundary_rhs, h->grid_b, kThreads, 0, M));
        h->launches += 1;
    }
    return halo_push(h, h->cur_x);      // x0 = c~: the first residual gathers the neighbours' rows
}

// pointers and scalars of step t (hydrodynamic slices t / t + 1 in slots s0 / s1)
static StepParams step_params(cwr_handle* h, int t, int s0, int s1) {
    const int n = h->n, E = h->E, K = h->K, Eg = std::max(1, h->topo.E_g), G = std::max(1, h->G);
    StepParams p;
    p.adv_t = h->d_adv + (size_t)s0 * E; p.cdiff_t = h->d_cdiff + (size_t)s0 * E;
    p.vol_t = h->d_vol + (size_t)s0 * n; p.vol_t1 = h->d_vol + (size_t)s1 * n;
    p.adv_t1 = h->d_adv + (size_t)s1 * E; p.cdiff_t1 = h->d_cdiff + (size_t)s1 * E;
    p.velg_t1 = h->d_velg + (size_t)s1 * Eg;
    p.flowg_t = h->d_flowg + (size_t)s0 * Eg;
    p.bc_t1 = h->d_bc + (size_t)(t + 1) * G * K;
    p.state_t = state_slot(h, t); p.state_t1 = state_slot(h, t + 1);
    p.dt = h->dt[t]; p.t = t; p.apply_ic = (t == 0);
    return p;
}

int cwr_step(cwr_handle* h, int t, cwr_step_info* info) {
    if (!h) return CWR_EINVAL;
    if (t < 0 || t + 1 >= h->T) FAIL(CWR_EINVAL, "cwr_step: t must satisfy 0 <= t < n_time - 1 (dt[n_time-1] is NaN)");
    if (t > h->computed_upto) FAIL(CWR_EINVAL, "cwr_step: c[t] has not been computed yet");
    if (!h->opt.keep_history && t < h->computed_upto - 1) FAIL(CWR_EINVAL, "cwr_step: c[t] no longer on the device");
    for (int k = 0; k < h->K; ++k)
        if (!h->inputs_set[k]) FAIL(CWR_EINVAL, "cwr_set_inputs has not been called for every constituent");
    const int s0 = find_slot(h, t), s1 = find_slot(h, t + 1);
    if (s0 < 0 || s1 < 0) FAIL(CWR_EINVAL, "hydrodynamic slices t and t+1 are not resident; call cwr_set_hydro");
    CK(cudaSetDevice(h->device));
    { int rcj = join_prefetch(h, s0); if (rcj) return rcj; rcj = join_prefetch(h, s1); if (rcj) return rcj; }
    const int64_t launches0 = h->launches;
    const StepParams p = step_params(h, t, s0, s1);
    DeviceModel& M = h->M;
    if (h->sp_ready) M.sp = const_cast<StepParams*>(h->sp_ready);      // (cwr_run, small-mesh path: uploaded with the run's other steps)
    else CK(launch_chain(h, k_set_step, 1, 1, 0, p, h->d_sp, M.ctl, h->world > 1 ? M.dd : (DdCtl*)nullptr));
    h->cur_x = p.state_t1;
    mark(h, CWR_FAM_ASSEMBLE);
    if (h->world > 1 && !h->attached) FAIL(CWR_EINVAL, "domain-decomposed handle: call cwr_dd_attach before stepping");
    const int nb_own = M.b_hi - M.b_lo;
    if (nb_own > 0) CK(launch_chain(h, k_boundary_diag, grid_for(nb_own, kThreads, h->max_grid), kThreads, 0, M));
    CK(launch_chain(h, k_assemble, grid_for(M.row_hi - M.row_lo, kThreads, h->max_grid), kThreads, 0, M));
    h->launches += 2 + (nb_own > 0);
    h->lhs_step = t;
    { int rc = build_rhs(h, t, 1); if (rc) return rc; }
    cwr_step_info local{};
    int status;
    if (h->small_path) status = solve_small(h, &local);
    else if (h->dc) {
        bool fell_back = false;
        status = solve_dc(h, &local, &fell_back);
        if (fell_back) {
            // the sweeps did not contract (not the M-matrix they assume): start again from c~ with BiCGSTAB
            ++h->fallbacks;
            const int cycles = h->h_ctl->iter, sweeps = h->h_ctl->sweeps_done;
            CK(cudaMemsetAsync(&M.ctl->all_done, 0, 2 * sizeof(int), h->stream));   // all_done, iter
            h->last_iters = 0;
            { int rc = build_rhs(h, t, 0); if (rc) return rc; }
            status = solve(h, &local);
            local.restarts += 1 + cycles;
            local.sweeps = sweeps;
        }
    } else status = solve(h, &local);
    if (status == CWR_ECUDA) return status;
    // transport.py:258-264: non-zero input_array[t+1] entries are re-imposed on the stored row -- ghost cells
    // are handled where they are read (k_mass_flux, k_extract_state); real cells (rare) are patched here.
    { int rc = patch_real_cells(h, t + 1, 0); if (rc) return rc; }
    // c[t+1] of the neighbours' boundary rows: the mass flux of a cut edge and the next cwr_get_state read them
    { int rc = halo_push(h, p.state_t1); if (rc) return rc; }
    if (M.want_flux) {
        mark(h, CWR_FAM_MASS_FLUX);
        KC_DISPATCH(h->KC, (launch_chain(h, k_mass_flux<KC, VEC>, h->grid_edges, kThreads, 0, M)));
        h->launches += 1;
        h->flux_step = t;
    }
    flush_profile(h);
    CK(cudaGetLastError());
    h->computed_upto = std::max(h->computed_upto, t + 1);
    if (!h->opt.keep_history) h->computed_upto = t + 1;
    local.n_launches = (int)(h->launches - launches0);
    if (info) *info = local;
    if (status != CWR_OK) {
        char buf[160];
        std::snprintf(buf, sizeof buf, "step %d: solver status %d after %d iterations (max relres %.3e)", t, status,
                      local.iterations, local.max_relres);
        h->err = buf;
    }
    return status;
}

int cwr_run(cwr_handle* h, int t_begin, int t_end, cwr_step_info* worst) {
    if (!h) return CWR_EINVAL;
    cwr_step_info w{}; w.status = CWR_OK;
    int rc_final = CWR_OK;
    if (h->small_path) {
        // every step is a fixed sequence of launches with the convergence loop on the device: queue all
        // of them, synchronise once, report the worst solver statistics over the run
        CK(cudaSetDevice(h->device));
        CK(cudaMemsetAsync(h->d_stats, 0, sizeof(SmallStats), h->stream));
        // the parameters of all the steps in one upload (their hydrodynamic slices are resident for the whole call: nothing
        // is uploaded in between); k_set_step once, for the control block
        bool ring = t_end > t_begin && t_begin >= 0 && t_end < h->T && !std::getenv("CWR_NO_SP_RING");
        h->sp_host.clear();
        for (int t = t_begin; ring && t < t_end; ++t) {
            const int s0 = find_slot(h, t), s1 = find_slot(h, t + 1);
            if (s0 < 0 || s1 < 0) ring = false;
            else h->sp_host.push_back(step_params(h, t, s0, s1));
        }
        if (ring) {
            const size_t cnt = h->sp_host.size();
            if (cnt > h->sp_ring_cap) {
                CK(cudaStreamSynchronize(h->stream));
                if (h->d_sp_ring) CK(cudaFree(h->d_sp_ring));
                h->d_sp_ring = nullptr; h->sp_ring_cap = 0;
                CK(cudaMalloc((void**)&h->d_sp_ring, (cnt + cnt / 2 + 16) * sizeof(StepParams)));
                h->sp_ring_cap = cnt + cnt / 2 + 16;
            }
            // (pageable source: the copy has left the host vector when the call returns)
            CK(cudaMemcpyAsync(h->d_sp_ring, h->sp_host.data(), cnt * sizeof(StepParams), cudaMemcpyHostToDevice, h->stream));
            CK(launch_chain(h, k_set_step, 1, 1, 0, h->sp_host[0], h->d_sp, h->M.ctl, (DdCtl*)nullptr));
            h->launches += 1;
        }
        h->in_run = true;
        int rc = CWR_OK;
        for (int t = t_begin; t < t_end && rc == CWR_OK; ++t) {
            cwr_step_info i{};
            h->sp_ready = ring ? h->d_sp_ring + (t - t_begin) : nullptr;
            rc = cwr_step(h, t, &i);
            w.n_launches += i.n_launches;
        }
        h->in_run = false;
        h->sp_ready = nullptr;
        h->M.sp = h->d_sp;
        if (ring && rc == CWR_OK)     // what a later call reads through M.sp (cwr_get_lhs / cwr_get_rhs): the last step's parameters
            CK(cudaMemcpyAsync(h->d_sp, h->d_sp_ring + (t_end - 1 - t_begin), sizeof(StepParams), cudaMemcpyDeviceToDevice, h->stream));
        if (rc != CWR_OK) return rc;
        const int n_launches = w.n_launches;
        rc = read_small_stats(h, &w);
        w.n_launches = n_launches;
        if (rc != CWR_ECUDA) h->iterations += (int64_t)(h->h_stats->sum_iterations / (unsigned long long)h->K);
        if (worst) *worst = w;
        return rc;
    }
    for (int t = t_begin; t < t_end; ++t) {
        cwr_step_info i{};
        int rc = cwr_step(h, t, &i);
        if (rc == CWR_EINVAL || rc == CWR_ECUDA) return rc;
        if (rc != CWR_OK && rc_final == CWR_OK) rc_final = rc;
        w.iterations = std::max(w.iterations, i.iterations);
        w.restarts = std::max(w.restarts, i.restarts);
        w.max_relres = std::max(w.max_relres, i.max_relres);
        w.n_launches += i.n_launches;
        if (i.status != CWR_OK) w.status = i.status;
    }
    if (worst) *worst = w;
    return rc_final;
}

// ------------------------------------------------------------------------------------------------
// outputs
// ------------------------------------------------------------------------------------------------
int cwr_get_state(cwr_handle* h, int k, int t, double* out) {
    if (!h) return CWR_EINVAL;
    if (!out) FAIL(CWR_EINVAL, "NULL array");
    if (k < 0 || k >= h->K) FAIL(CWR_EINVAL, "constituent index out of range");
    int rc = state_available(h, t);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    rc = ensure_stage(h, (size_t)h->F * 8);
    if (rc) return rc;
    const double* bc_t = (t >= 1 && h->G > 0) ? h->d_bc + (size_t)t * h->G * h->K : nullptr;
    k_extract_state<<<grid_for(h->F, kThreads, h->max_grid), kThreads, 0, h->stream>>>(
        (double*)h->d_stage, state_slot(h, t), bc_t, h->d_new_of_old, h->n, h->F, h->K, k);
    h->launches += 1;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, h->d_stage, (size_t)h->F * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    if (t == 0 && !h->initial_row[k].empty())   // row 0 = the IC row: zeros (not NaN) where unset
        std::copy(h->initial_row[k].begin() + h->n, h->initial_row[k].end(), out + h->n);
    return CWR_OK;
}

int cwr_get_state_all(cwr_handle* h, int t, double* out) {
    if (!h) return CWR_EINVAL;
    if (!out) FAIL(CWR_EINVAL, "NULL array");
    int rc = state_available(h, t);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    const size_t nK = (size_t)h->n * h->K;
    rc = ensure_stage(h, nK * 8);
    if (rc) return rc;
    launch_extract(h, (double*)h->d_stage, state_slot(h, t), h->d_new_of_old, h->n, (size_t)h->n);
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, h->d_stage, nK * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return CWR_OK;
}

int cwr_get_state_rows(cwr_handle* h, int t, double* const* rows) {
    if (!h) return CWR_EINVAL;
    if (!rows) FAIL(CWR_EINVAL, "NULL array");
    int rc = state_available(h, t);
    if (rc) return rc;
    CK(cudaSetDevice(h->device));
    const size_t nK = (size_t)h->n * h->K;
    rc = ensure_stage(h, nK * 8);
    if (rc) return rc;
    launch_extract(h, (double*)h->d_stage, state_slot(h, t), h->d_new_of_old, h->n, (size_t)h->n);
    CK(cudaGetLastError());
    for (int k = 0; k < h->K; ++k) {
        if (!rows[k]) continue;
        CK(cudaMemcpyAsync(rows[k], (const double*)h->d_stage + (size_t)k * h->n, (size_t)h->n * 8, cudaMemcpyDeviceToHost, h->stream));
    }
    CK(cudaStreamSynchronize(h->stream));
    return CWR_OK;
}

int cwr_fetch_async(cwr_handle* h, int t, double* const* state_rows, double* const* adv_rows, double* const* diff_rows,
                    double* const* tot_rows) {
    if (!h) return CWR_EINVAL;
    int rc = state_available(h, t);
    if (rc) return rc;
    const bool want_flux = adv_rows || diff_rows || tot_rows;
    if (want_flux && !h->M.want_flux) FAIL(CWR_EINVAL, "mass flux disabled (options.mass_flux = 0)");
    if (want_flux && t - 1 != h->flux_step) FAIL(CWR_EINVAL, "only the most recent step's mass fluxes are on the device");
    CK(cudaSetDevice(h->device));
    if (!h->out_stream) {
        CK(cudaStreamCreateWithFlags(&h->out_stream, cudaStreamNonBlocking));
        for (int i = 0; i < 2; ++i) {
            CK(cudaEventCreateWithFlags(&h->ev_extract[i], cudaEventDisableTiming));
            CK(cudaEventCreateWithFlags(&h->ev_copied[i], cudaEventDisableTiming));
        }
    }
    const int slot = h->out_next;
    h->out_next ^= 1;
    const size_t nK = (size_t)h->n * h->K, EK = (size_t)h->E * h->K;
    const size_t need = (nK + (want_flux ? 3 * EK : 0)) * sizeof(double);
    // the slot's previous copies (two fetches ago) must have left it
    if (h->out_pending[slot]) { CK(cudaEventSynchronize(h->ev_copied[slot])); h->out_pending[slot] = false; }
    if (need > h->out_bytes[slot]) {
        if (h->d_out[slot]) { CK(cudaFree(h->d_out[slot])); h->d_out[slot] = nullptr; h->out_bytes[slot] = 0; }
        if (cudaMalloc((void**)&h->d_out[slot], need) != cudaSuccess) { cudaGetLastError(); FAIL(CWR_ENOMEM, "no device memory for the output staging slot"); }
        h->out_bytes[slot] = need;
    }
    double* st = h->d_out[slot];
    if (state_rows) launch_extract(h, st, state_slot(h, t), h->d_new_of_old, h->n, (size_t)h->n);
    if (want_flux)
        for (int w = 0; w < 3; ++w)
            launch_extract(h, st + nK + (size_t)w * EK, h->M.flux + (size_t)w * EK, h->d_einv, h->E, (size_t)h->E);
    CK(cudaGetLastError());
    CK(cudaEventRecord(h->ev_extract[slot], h->stream));
    CK(cudaStreamWaitEvent(h->out_stream, h->ev_extract[slot], 0));
    for (int k = 0; k < h->K; ++k) {
        if (state_rows && state_rows[k])
            CK(cudaMemcpyAsync(state_rows[k], st + (size_t)k * h->n, (size_t)h->n * 8, cudaMemcpyDeviceToHost, h->out_stream));
        double* const* fr[3] = {adv_rows, diff_rows, tot_rows};
        for (int w = 0; w < 3; ++w)
            if (fr[w] && fr[w][k])
                CK(cudaMemcpyAsync(fr[w][k], st + nK + (size_t)w * EK + (size_t)k * h->E, (size_t)h->E * 8, cudaMemcpyDeviceToHost, h->out_stream));
    }
    CK(cudaEventRecord(h->ev_copied[slot], h->out_stream));
    h->out_pending[slot] = true;
    return CWR_OK;
}

int cwr_fetch_wait(cwr_handle* h) {
    if (!h) return CWR_EINVAL;
    CK(cudaSetDevice(h->device));
    for (int i = 0; i < 2; ++i)
        if (h->out_pending[i]) { CK(cudaEventSynchronize(h->ev_copied[i])); h->out_pending[i] = false; }
    return CWR_OK;
}

int cwr_host_register(void* p, size_t bytes) {
    if (!p || bytes == 0) return CWR_EINVAL;
    cudaError_t e = cudaHostRegister(p, bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess) { g_create_error = std::string("cudaHostRegister: ") + cudaGetErrorString(e); cudaGetLastError(); return CWR_ECUDA; }
    return CWR_OK;
}

int cwr_host_unregister(void* p) {
    if (!p) return CWR_EINVAL;
    cudaError_t e = cudaHostUnregister(p);
    if (e != cudaSuccess) { cudaGetLastError(); return CWR_ECUDA; }
    return CWR_OK;
}

int cwr_get_mass_flux(cwr_handle* h, int k, int t, double* adv, double* diff, double* tot) {
    if (!h) return CWR_EINVAL;
    if (k < 0 || k >= h->K) FAIL(CWR_EINVAL, "constituent index out of range");
    if (!h->M.want_flux) FAIL(CWR_EINVAL, "mass flux disabled (options.mass_flux = 0)");
    if (t != h->flux_step) FAIL(CWR_EINVAL, "only the most recent step's mass fluxes are on the device");
    CK(cudaSetDevice(h->device));
    int rc = ensure_stage(h, (size_t)h->E * 8);
    if (rc) return rc;
    double* outs[3] = {adv, diff, tot};
    for (int w = 0; w < 3; ++w) {
        if (!outs[w]) continue;
        k_extract_flux<<<grid_for(h->E, kThreads, h->max_grid), kThreads, 0, h->stream>>>(
            (double*)h->d_stage, h->M.flux + (size_t)w * h->E * h->K, h->d_einv, h->E, h->K, k);
        h->launches += 1;
        CK(cudaMemcpyAsync(outs[w], h->d_stage, (size_t)h->E * 8, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    CK(cudaGetLastError());
    return CWR_OK;
}

int cwr_get_flux_sums(cwr_handle* h, int k, double* total_sum, double* in_sum, double* out_sum) {
    if (!h) return CWR_EINVAL;
    if (k < 0 || k >= h->K) FAIL(CWR_EINVAL, "constituent index out of range");
    if (!h->M.want_flux) FAIL(CWR_EINVAL, "mass flux disabled (options.mass_flux = 0)");
    CK(cudaSetDevice(h->device));
    const int Eg = h->topo.E_g, Ei = h->topo.E_int, K = h->K;
    std::vector<double> host((size_t)3 * std::max(1, Eg) * K);
    CK(cudaMemcpyAsync(host.data(), h->M.bsum, host.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    double* outs[3] = {total_sum, in_sum, out_sum};
    for (int w = 0; w < 3; ++w) {
        if (!outs[w]) continue;
        std::fill(outs[w], outs[w] + h->E, 0.0);
        for (int g = 0; g < Eg; ++g) outs[w][h->topo.eperm[Ei + g]] = host[((size_t)w * Eg + g) * K + k];
    }
    return CWR_OK;
}

int cwr_get_volume_sums(cwr_handle* h, double* total_sum, double* in_sum, double* out_sum) {
    if (!h) return CWR_EINVAL;
    if (!h->M.want_flux) FAIL(CWR_EINVAL, "mass flux disabled (options.mass_flux = 0)");
    CK(cudaSetDevice(h->device));
    const int Eg = h->topo.E_g, Ei = h->topo.E_int;
    std::vector<double> host((size_t)3 * std::max(1, Eg));
    CK(cudaMemcpyAsync(host.data(), h->M.vsum, host.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    double* outs[3] = {total_sum, in_sum, out_sum};
    for (int w = 0; w < 3; ++w) {
        if (!outs[w]) continue;
        std::fill(outs[w], outs[w] + h->E, 0.0);
        for (int g = 0; g < Eg; ++g) outs[w][h->topo.eperm[Ei + g]] = host[(size_t)w * Eg + g];
    }
    return CWR_OK;
}

int cwr_set_kinetics(cwr_handle* h, const double* decay, const double* theta, const double* yields, int temperature_k,
                     double temperature_c) {
    if (!h) return CWR_EINVAL;
    const int K = h->K;
    if (!decay) { h->kin_on = false; h->kin_srcs = 0; h->kin_facs = 0; h->kin_depth = false; h->kin_forced = false; return CWR_OK; }
    for (int k = 0; k < K; ++k) {
        if (!std::isfinite(decay[k]) || decay[k] < 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics: decay rates must be finite and >= 0");
        if (theta && (!std::isfinite(theta[k]) || theta[k] <= 0.0)) FAIL(CWR_EINVAL, "cwr_set_kinetics: theta must be finite and > 0");
    }
    if (yields)
        for (int j = 0; j < K; ++j)
            for (int k = 0; k < K; ++k) {
                const double y = yields[(size_t)j * K + k];
                if (!std::isfinite(y)) FAIL(CWR_EINVAL, "cwr_set_kinetics: yields must be finite");
                if (j == k && y != 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics: a constituent cannot yield itself");
            }
    if (temperature_k < -1 || temperature_k >= K) FAIL(CWR_EINVAL, "cwr_set_kinetics: temperature constituent out of range");
    if (temperature_k < 0 && !std::isfinite(temperature_c)) FAIL(CWR_EINVAL, "cwr_set_kinetics: temperature must be finite");
    if (temperature_k >= 0) {
        if (decay[temperature_k] != 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics: the temperature constituent cannot decay");
        for (int k = 0; yields && k < K; ++k)
            if (yields[(size_t)temperature_k * K + k] != 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics: the temperature constituent cannot receive a yield");
    }
    // topological order of the yield graph (k -> j where yields[j, k] != 0), smallest index first among the ready ones
    std::vector<int> indeg(K, 0), order;
    for (int j = 0; yields && j < K; ++j)
        for (int k = 0; k < K; ++k) indeg[j] += yields[(size_t)j * K + k] != 0.0;
    std::vector<uint8_t> done(K, 0);
    for (int round = 0; round < K; ++round) {
        int k = 0;
        while (k < K && (done[k] || indeg[k] != 0)) ++k;
        if (k == K) FAIL(CWR_EINVAL, "cwr_set_kinetics: the yield graph has a cycle");
        done[k] = 1;
        order.push_back(k);
        for (int j = 0; yields && j < K; ++j) indeg[j] -= yields[(size_t)j * K + k] != 0.0;
    }
    // a constituent that does not decay forms no loss (and so yields nothing): only the decaying ones are steps
    std::vector<KinStep> steps;
    std::vector<KinYield> ylist;
    for (int k : order) {
        if (decay[k] == 0.0) continue;
        KinStep s{};
        s.col = k; s.decay = decay[k]; s.log_theta = theta ? std::log(theta[k]) : 0.0;
        s.y_begin = (int)ylist.size();
        for (int j = 0; yields && j < K; ++j) {
            const double y = yields[(size_t)j * K + k];
            if (y != 0.0) { KinYield e{}; e.col = j; e.y = y; ylist.push_back(e); }
        }
        s.y_end = (int)ylist.size();
        steps.push_back(s);
    }
    CK(cudaSetDevice(h->device));
    if (!h->d_kin_state) {
        for (auto* fn : {k_react<false>, k_react<true>, k_react<true, true>, k_react<false, false, true>,
                         k_react<true, false, true>, k_react<true, true, true>}) {
            cudaFuncAttributes fa{};
            CK(cudaFuncGetAttributes(&fa, fn));
            if (fa.sharedSizeBytes > kReactStaticSmem)
                FAIL(CWR_ECUDA, "k_react: static shared memory exceeds what its tile sizing reserves");
        }
        // the grid of every instantiation (the factored ones may hold fewer CTAs per SM; their CTAs need not be co-resident)
        int occ = 0;
        CK(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_react<false>, kThreads, react_smem_bytes(K)));
        h->kin_grid_max = h->num_sms * std::max(1, occ);
        CK(dalloc(h, &h->d_kin_steps, (size_t)K));
        CK(dalloc(h, &h->d_kin_yields, (size_t)K * K));
        CK(dalloc(h, &h->d_kin_partials, (size_t)K * h->kin_grid_max));
        CK(dalloc(h, &h->d_kin_state, 1));
        CK(dalloc(h, &h->d_kin_srcs, (size_t)K));
        CK(dalloc(h, &h->d_kin_facs, (size_t)4 * K * K));      // at most (decay | source) x column x factor column x kind
        CK(dalloc(h, &h->d_kin_fptr, (size_t)2 * K + 1));
        CK(dalloc(h, &h->d_kin_fptr0, (size_t)2 * K + 1));
        CK(dalloc(h, &h->d_kin_dflag, (size_t)2 * K));
        CK(dalloc(h, &h->d_kin_area, (size_t)h->n));
        CK(cudaMemsetAsync(h->d_kin_state, 0, sizeof(KinState), h->stream));
        CK(cudaMemsetAsync(h->d_kin_fptr0, 0, ((size_t)2 * K + 1) * sizeof(int), h->stream));
    }
    // stream-ordered: steps queued before this call still read the previous parameters (pageable sources: the copies
    // have left the host vectors when the calls return)
    if (!steps.empty()) CK(cudaMemcpyAsync(h->d_kin_steps, steps.data(), steps.size() * sizeof(KinStep), cudaMemcpyHostToDevice, h->stream));
    if (!ylist.empty()) CK(cudaMemcpyAsync(h->d_kin_yields, ylist.data(), ylist.size() * sizeof(KinYield), cudaMemcpyHostToDevice, h->stream));
    h->kin_steps = (int)steps.size();
    h->kin_temp_k = temperature_k;
    h->kin_temp_c = temperature_k < 0 ? temperature_c : 20.0;
    h->kin_on = true;
    h->kin_srcs = 0;
    h->kin_facs = 0;
    h->kin_depth = false;
    h->kin_forced = false;
    h->kin_decay_h.assign(decay, decay + K);
    h->kin_yields_h.assign((size_t)K * K, 0.0);
    if (yields) h->kin_yields_h.assign(yields, yields + (size_t)K * K);
    h->kin_step_of.assign(K, -1);
    for (size_t p = 0; p < steps.size(); ++p) h->kin_step_of[steps[p].col] = (int)p;
    h->kin_source_h.assign(K, 0.0);
    h->kin_exchange_h.assign(K, 0.0);
    h->kin_src_of.assign(K, -1);
    h->kin_kind_h.assign(K, 0);
    return CWR_OK;
}

int cwr_set_kinetics_sources(cwr_handle* h, const double* source_per_day, const double* source_theta, const double* exchange_per_day,
                             const double* exchange_theta, const double* equilibrium, const int* equilibrium_kind) {
    if (!h) return CWR_EINVAL;
    const int K = h->K;
    if (!h->kin_on) FAIL(CWR_EINVAL, "cwr_set_kinetics_sources: call cwr_set_kinetics first");
    if (!source_per_day && !exchange_per_day) {
        h->kin_srcs = 0; h->kin_facs = 0; h->kin_depth = false; h->kin_forced = false;
        h->kin_source_h.assign(K, 0.0); h->kin_exchange_h.assign(K, 0.0); h->kin_src_of.assign(K, -1); h->kin_kind_h.assign(K, 0);
        return CWR_OK;
    }
    if (exchange_per_day && !equilibrium) FAIL(CWR_EINVAL, "cwr_set_kinetics_sources: exchange needs an equilibrium array");
    for (int k = 0; k < K; ++k) {
        const double s = source_per_day ? source_per_day[k] : 0.0, e = exchange_per_day ? exchange_per_day[k] : 0.0;
        const int kind = equilibrium_kind ? equilibrium_kind[k] : 0;
        if (!std::isfinite(s)) FAIL(CWR_EINVAL, "cwr_set_kinetics_sources: sources must be finite");
        if (source_theta && (!std::isfinite(source_theta[k]) || source_theta[k] <= 0.0))
            FAIL(CWR_EINVAL, "cwr_set_kinetics_sources: source_theta must be finite and > 0");
        if (exchange_theta && (!std::isfinite(exchange_theta[k]) || exchange_theta[k] <= 0.0))
            FAIL(CWR_EINVAL, "cwr_set_kinetics_sources: exchange_theta must be finite and > 0");
        if (!std::isfinite(e) || e < 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics_sources: exchange rates must be finite and >= 0");
        if (kind != 0 && kind != 1) FAIL(CWR_EINVAL, "cwr_set_kinetics_sources: equilibrium_kind must be 0 (constant) or 1 (oxygen saturation)");
        if (kind == 0 && e > 0.0 && !std::isfinite(equilibrium[k]))
            FAIL(CWR_EINVAL, "cwr_set_kinetics_sources: a constant equilibrium must be finite");
        if (kind == 1 && k == h->kin_temp_k)
            FAIL(CWR_EINVAL, "cwr_set_kinetics_sources: the temperature constituent cannot relax toward oxygen saturation");
    }
    // only the columns with a term are listed; the equilibrium of a column without exchange is never read
    std::vector<KinSrc> list;
    int o2 = 0;
    for (int k = 0; k < K; ++k) {
        const double s = source_per_day ? source_per_day[k] : 0.0, e = exchange_per_day ? exchange_per_day[k] : 0.0;
        if (s == 0.0 && e == 0.0) continue;
        KinSrc c{};
        c.col = k;
        c.kind = e > 0.0 && equilibrium_kind ? equilibrium_kind[k] : 0;
        c.source = s; c.log_source_theta = source_theta ? std::log(source_theta[k]) : 0.0;
        c.exchange = e; c.log_exchange_theta = exchange_theta ? std::log(exchange_theta[k]) : 0.0;
        c.equilibrium = e > 0.0 && c.kind == 0 ? equilibrium[k] : 0.0;
        o2 |= c.kind;
        list.push_back(c);
    }
    CK(cudaSetDevice(h->device));
    // at a constant temperature the coefficients take shared memory beyond the tile's 48 KB (react_src_smem_bytes); the
    // limit is the same for every handle (the attribute is the kernel's, not the handle's)
    if (h->kin_temp_k < 0 && !list.empty())
        for (auto* fn : {k_react<false>, k_react<true>, k_react<true, true>})
            CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)(kReactSmemLimit - kReactStaticSmem + react_src_smem_bytes(kMaxK, -1))));
    if (!list.empty()) CK(cudaMemcpyAsync(h->d_kin_srcs, list.data(), list.size() * sizeof(KinSrc), cudaMemcpyHostToDevice, h->stream));
    h->kin_srcs = (int)list.size();
    h->kin_src_o2 = o2;
    h->kin_facs = 0;
    h->kin_depth = false;
    h->kin_forced = false;
    h->kin_source_h.assign(K, 0.0);
    h->kin_exchange_h.assign(K, 0.0);
    h->kin_src_of.assign(K, -1);
    h->kin_kind_h.assign(K, 0);
    for (size_t p = 0; p < list.size(); ++p) {
        h->kin_source_h[list[p].col] = list[p].source;
        h->kin_exchange_h[list[p].col] = list[p].exchange;
        h->kin_src_of[list[p].col] = (int)p;
        h->kin_kind_h[list[p].col] = list[p].kind;
    }
    return CWR_OK;
}

int cwr_set_kinetics_limits(cwr_handle* h, int n, const int* process, const int* column, const int* factor_column,
                            const int* factor_kind, const double* half_saturation) {
    if (!h) return CWR_EINVAL;
    const int K = h->K;
    if (!h->kin_on) FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: call cwr_set_kinetics first");
    if (n < 0) FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: n must be >= 0");
    if (n == 0 || !process || !column || !factor_column || !factor_kind || !half_saturation) { h->kin_facs = 0; return CWR_OK; }
    std::vector<long long> seen;
    for (int i = 0; i < n; ++i) {
        const int pr = process[i], k = column[i], j = factor_column[i], kind = factor_kind[i];
        const double half = half_saturation[i];
        if (pr != 0 && pr != 1) FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: process must be 0 (decay) or 1 (source)");
        if (kind != 0 && kind != 1) FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: factor_kind must be 0 (limitation) or 1 (inhibition)");
        if (k < 0 || k >= K || j < 0 || j >= K) FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: column index out of range");
        if (!std::isfinite(half) || half <= 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: half-saturations must be finite and > 0");
        if (pr == 0 && h->kin_decay_h[k] == 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: a decay factor on a column that does not decay");
        if (pr == 1 && h->kin_source_h[k] == 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: a source factor on a column without a source");
        if (pr == 0 && j == k) FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: a decay cannot be limited or inhibited by its own column");
        if (pr == 1 && j == k && (kind != 0 || h->kin_source_h[k] >= 0.0))
            FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: only a sink (source < 0) can be limited by its own column");
        seen.push_back((((long long)pr * K + k) * K + j) * 2 + kind);
    }
    std::sort(seen.begin(), seen.end());
    if (std::adjacent_find(seen.begin(), seen.end()) != seen.end())
        FAIL(CWR_EINVAL, "cwr_set_kinetics_limits: the same (process, column, factor column, kind) given twice");
    // grouped per process (the decay steps in their order, then the source columns in theirs), each in the order given
    const int n_proc = h->kin_steps + h->kin_srcs;
    std::vector<std::vector<KinFac>> per(n_proc);
    for (int i = 0; i < n; ++i) {
        const int k = column[i], j = factor_column[i];
        const int q = process[i] == 0 ? h->kin_step_of[k] : h->kin_steps + h->kin_src_of[k];
        KinFac a{};
        a.col = j; a.kind = factor_kind[i]; a.half = half_saturation[i];
        const double y = h->kin_yields_h[(size_t)j * K + k];
        a.use = process[i] == 0 && a.kind == 0 && y < 0.0 ? -y : 0.0;
        per[q].push_back(a);
    }
    std::vector<KinFac> list;
    std::vector<int> ptr(1, 0);
    for (const auto& v : per) { list.insert(list.end(), v.begin(), v.end()); ptr.push_back((int)list.size()); }
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(h->d_kin_facs, list.data(), list.size() * sizeof(KinFac), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_kin_fptr, ptr.data(), ptr.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    h->kin_facs = (int)list.size();
    return CWR_OK;
}

int cwr_set_kinetics_depth(cwr_handle* h, const double* cell_area, double min_depth, const int* decay_per_depth,
                           const int* source_per_depth, const int* exchange_per_depth) {
    if (!h) return CWR_EINVAL;
    const int K = h->K;
    if (!h->kin_on) FAIL(CWR_EINVAL, "cwr_set_kinetics_depth: call cwr_set_kinetics first");
    const int* flags[3] = {decay_per_depth, source_per_depth, exchange_per_depth};
    bool any = false;
    for (const int* f : flags)
        for (int k = 0; f && k < K; ++k) {
            if (f[k] != 0 && f[k] != 1) FAIL(CWR_EINVAL, "cwr_set_kinetics_depth: flags must be 0 or 1");
            any |= f[k] == 1;
        }
    if (!any) { h->kin_depth = false; return CWR_OK; }
    const double* rate[3] = {h->kin_decay_h.data(), h->kin_source_h.data(), h->kin_exchange_h.data()};
    for (int w = 0; w < 3; ++w)
        for (int k = 0; flags[w] && k < K; ++k)
            if (flags[w][k] && rate[w][k] == 0.0)
                FAIL(CWR_EINVAL, "cwr_set_kinetics_depth: a depth flag on a process whose rate is 0");
    if (!cell_area) FAIL(CWR_EINVAL, "cwr_set_kinetics_depth: depth flags need the cell areas");
    if (!std::isfinite(min_depth) || min_depth <= 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics_depth: min_depth must be finite and > 0");
    for (int i = 0; i < h->n; ++i) {
        const double a = cell_area[h->topo.old_of_new[i]];
        if (!std::isfinite(a) || a <= 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics_depth: cell areas must be finite and > 0");
    }
    // per process, numbered as d_kin_fptr: the decay steps in their order, then the source columns in theirs
    std::vector<int> dflag(h->kin_steps + h->kin_srcs, 0);
    for (int k = 0; k < K; ++k) {
        if (h->kin_step_of[k] >= 0 && decay_per_depth) dflag[h->kin_step_of[k]] = decay_per_depth[k];
        if (h->kin_src_of[k] >= 0)
            dflag[h->kin_steps + h->kin_src_of[k]] = (source_per_depth ? source_per_depth[k] : 0) |
                                                     (exchange_per_depth ? exchange_per_depth[k] : 0) << 1;
    }
    CK(cudaSetDevice(h->device));
    h->kin_area_h.assign(cell_area, cell_area + h->F);
    int rc = upload_kin_area(h);
    if (rc) return rc;
    CK(cudaMemcpyAsync(h->d_kin_dflag, dflag.data(), dflag.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    h->kin_min_depth = min_depth;
    h->kin_depth = true;
    return CWR_OK;
}

int cwr_set_kinetics_forcing(cwr_handle* h, int n, int n_time, const int* target, const int* column, const double* values) {
    if (!h) return CWR_EINVAL;
    const int K = h->K, T = h->T;
    if (!h->kin_on) FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: call cwr_set_kinetics first");
    if (n < 0) FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: n must be >= 0");
    if (n == 0) { h->kin_forced = false; return CWR_OK; }
    if (n_time != T) FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: n_time must be the handle's n_time");
    if (!target || !column || !values) FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: NULL array with n > 0");
    const double* rate[5] = {nullptr, nullptr, h->kin_decay_h.data(), h->kin_source_h.data(), h->kin_exchange_h.data()};
    std::vector<int> seen;
    for (int i = 0; i < n; ++i) {
        const int g = target[i], k = column[i];
        if (g < CWR_FORCE_TEMPERATURE || g > CWR_FORCE_EXCHANGE_SCALE) FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: unknown target");
        if (g == CWR_FORCE_TEMPERATURE) {
            if (k != -1) FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: the temperature series takes column -1");
            if (h->kin_temp_k >= 0)
                FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: a temperature series while a temperature constituent is set");
        } else if (k < 0 || k >= K) FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: column index out of range");
        seen.push_back(g * (K + 1) + k + 1);
        const double* v = values + (size_t)i * T;
        for (int t = 0; t < T; ++t) {
            if (!std::isfinite(v[t])) FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: a series value is not finite");
            if (g >= CWR_FORCE_DECAY_SCALE && v[t] < 0.0) FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: a scale is negative");
        }
        if (g >= CWR_FORCE_DECAY_SCALE && rate[g][k] == 0.0)
            FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: a scale on a process whose rate is 0");
        if (g == CWR_FORCE_EQUILIBRIUM && h->kin_exchange_h[k] == 0.0)
            FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: an equilibrium series on a column without exchange");
        if (g == CWR_FORCE_EQUILIBRIUM && h->kin_kind_h[k] != 0)
            FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: an equilibrium series on a column that relaxes toward oxygen saturation");
    }
    std::sort(seen.begin(), seen.end());
    if (std::adjacent_find(seen.begin(), seen.end()) != seen.end())
        FAIL(CWR_EINVAL, "cwr_set_kinetics_forcing: the same (target, column) given twice");
    // the series row of every forced parameter, numbered as k_react reads them (-1: not forced)
    std::vector<int> fmap(1 + h->kin_steps + 3 * h->kin_srcs, -1);
    for (int i = 0; i < n; ++i) {
        const int g = target[i], k = column[i];
        if (g == CWR_FORCE_TEMPERATURE) fmap[0] = i;
        else if (g == CWR_FORCE_DECAY_SCALE) fmap[1 + h->kin_step_of[k]] = i;
        else fmap[1 + h->kin_steps + 3 * h->kin_src_of[k] + (g == CWR_FORCE_SOURCE_SCALE ? 0 : g == CWR_FORCE_EXCHANGE_SCALE ? 1 : 2)] = i;
    }
    CK(cudaSetDevice(h->device));
    if (!h->d_kin_force) {
        CK(dalloc(h, &h->d_kin_force, (size_t)(1 + 4 * K) * T));
        CK(dalloc(h, &h->d_kin_fmap, (size_t)1 + 4 * K));
        h->M.kin_force = h->d_kin_force; h->M.kin_fmap = h->d_kin_fmap; h->M.n_time = T;
        // the forced source columns take shared memory beyond the coefficients (react_force_smem_bytes)
        for (auto* fn : {k_react<false, false, true>, k_react<true, false, true>, k_react<true, true, true>})
            CK(cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                    (int)(kReactSmemLimit - kReactStaticSmem + react_src_smem_bytes(kMaxK, -1) +
                                          react_force_smem_bytes(kMaxK))));
    }
    // stream-ordered, from host copies: steps queued before this call still read the previous series
    std::vector<double> table(values, values + (size_t)n * T);
    CK(cudaMemcpyAsync(h->d_kin_force, table.data(), table.size() * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    CK(cudaMemcpyAsync(h->d_kin_fmap, fmap.data(), fmap.size() * sizeof(int), cudaMemcpyHostToDevice, h->stream));
    h->kin_forced = true;
    return CWR_OK;
}

int cwr_get_reaction_mass(cwr_handle* h, int k, double* total) {
    if (!h) return CWR_EINVAL;
    if (!total) FAIL(CWR_EINVAL, "NULL output");
    if (k < 0 || k >= h->K) FAIL(CWR_EINVAL, "constituent index out of range");
    *total = 0.0;
    if (!h->d_kin_state) return CWR_OK;
    CK(cudaSetDevice(h->device));
    CK(cudaMemcpyAsync(total, &h->d_kin_state->mass[k], sizeof(double), cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    return CWR_OK;
}

int cwr_mass_totals_at(cwr_handle* h, int k, int t_start, int t_end, cwr_mass_totals* out) {
    if (!h) return CWR_EINVAL;
    if (!out) FAIL(CWR_EINVAL, "NULL output");
    if (k < 0 || k >= h->K) FAIL(CWR_EINVAL, "constituent index out of range");
    CK(cudaSetDevice(h->device));
    int ts[2] = {t_start, t_end};
    double res[2][2];
    int rc = ensure_stage(h, 64 + 16 * kMassBlocks);
    if (rc) return rc;
    double* d_out = (double*)h->d_stage;
    unsigned* d_ticket = (unsigned*)(d_out + 2);
    double* d_partial = d_out + 8;
    CK(cudaMemsetAsync(d_ticket, 0, sizeof(unsigned), h->stream));
    for (int i = 0; i < 2; ++i) {
        rc = state_available(h, ts[i]);
        if (rc) return rc;
        const int s = find_slot(h, ts[i]);
        if (s < 0) FAIL(CWR_EINVAL, "volume slice not resident for mass totals");
        { int rcj = join_prefetch(h, s); if (rcj) return rcj; }
        k_mass_total<<<grid_for(h->M.row_hi - h->M.row_lo, kThreads, kMassBlocks), kThreads, 0, h->stream>>>(
            h->d_vol + (size_t)s * h->n, state_slot(h, ts[i]), h->M.row_lo, h->M.row_hi, h->K, k, d_partial, d_ticket, d_out);
        h->launches += 1;
        CK(cudaMemcpyAsync(res[i], d_out, 16, cudaMemcpyDeviceToHost, h->stream));
        CK(cudaStreamSynchronize(h->stream));
    }
    out->vol_start = res[0][0]; out->mass_start = res[0][1]; out->vol_end = res[1][0]; out->mass_end = res[1][1];
    return CWR_OK;
}

int cwr_get_lhs(cwr_handle* h, int64_t* nnz, int32_t* indptr, int32_t* indices, double* data) {
    if (!h) return CWR_EINVAL;
    const Topology& tp = h->topo;
    // merged pattern size (duplicate (row, col) pairs collapse, as csr_matrix sums them)
    const int n = h->n;
    std::vector<std::vector<std::pair<int32_t, int32_t>>> rows(n);   // reference row -> (reference col, slot or -1 for diag)
    for (int i = 0; i < n; ++i) {
        auto& r = rows[tp.old_of_new[i]];
        r.emplace_back(tp.old_of_new[i], -1 - i);
        for (int j = tp.rowptr[i]; j < tp.rowptr[i + 1]; ++j)      // value index = ELL position of CSR slot j
            r.emplace_back(tp.old_of_new[tp.col[j]], (int32_t)((size_t)i * tp.W + (j - tp.rowptr[i])));
    }
    int64_t total = 0;
    for (auto& r : rows) {
        std::sort(r.begin(), r.end());
        int32_t last = -1;
        for (auto& pr : r) if (pr.first != last) { ++total; last = pr.first; }
    }
    if (nnz) *nnz = total;
    if (!indptr || !indices || !data) return CWR_OK;
    if (h->lhs_step < 0) FAIL(CWR_EINVAL, "no LHS assembled yet");
    CK(cudaSetDevice(h->device));
    std::vector<double> val((size_t)n * tp.W), diag(n);
    CK(cudaMemcpyAsync(val.data(), h->M.val, val.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(diag.data(), h->M.diag, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    int64_t pos = 0;
    for (int r0 = 0; r0 < n; ++r0) {
        indptr[r0] = (int32_t)pos;
        const int i = tp.new_of_old[r0];
        int32_t last = -1;
        for (auto& pr : rows[r0]) {
            const double v = pr.second < 0 ? diag[i] : val[pr.second] * diag[i];
            if (pr.first == last) data[pos - 1] += v;
            else { indices[pos] = pr.first; data[pos] = v; ++pos; last = pr.first; }
        }
    }
    indptr[n] = (int32_t)pos;
    return CWR_OK;
}

int cwr_get_rhs(cwr_handle* h, int k, double* b) {
    if (!h) return CWR_EINVAL;
    if (!b) FAIL(CWR_EINVAL, "NULL array");
    if (k < 0 || k >= h->K) FAIL(CWR_EINVAL, "constituent index out of range");
    if (h->lhs_step < 0) FAIL(CWR_EINVAL, "no step taken yet");
    CK(cudaSetDevice(h->device));
    const int n = h->n, K = h->K;
    std::vector<double> bs((size_t)n * K), diag(n);
    CK(cudaMemcpyAsync(bs.data(), h->M.b, bs.size() * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaMemcpyAsync(diag.data(), h->M.diag, (size_t)n * 8, cudaMemcpyDeviceToHost, h->stream));
    CK(cudaStreamSynchronize(h->stream));
    for (int r0 = 0; r0 < n; ++r0) {
        const int i = h->topo.new_of_old[r0];
        b[r0] = bs[(size_t)i * K + k] * diag[i];
    }
    return CWR_OK;
}

int cwr_get_permutation(cwr_handle* h, int32_t* new_of_old) {
    if (!h) return CWR_EINVAL;
    if (!new_of_old) FAIL(CWR_EINVAL, "NULL array");
    std::copy(h->topo.new_of_old.begin(), h->topo.new_of_old.end(), new_of_old);
    return CWR_OK;
}

int cwr_order_cells(int n_real, int n_face, int n_edge, const int32_t* f1, const int32_t* f2, int reorder, int n_colors,
                    const float* flow_hint, int n_parts, int32_t* new_of_old, int32_t* color_ptr, int* n_colors_out,
                    int* n_levels, int32_t* part_ptr, int32_t* n_send) {
    if (!f1 || !f2 || !new_of_old) return CWR_EINVAL;
    Topology t;
    const std::string terr = build_topology(n_real, n_face, n_edge, f1, f2, reorder != 0, n_colors, flow_hint, std::max(1, n_parts), t);
    if (!terr.empty()) { g_create_error = terr; return CWR_EINVAL; }
    std::copy(t.new_of_old.begin(), t.new_of_old.end(), new_of_old);
    if (color_ptr) std::copy(t.color_ptr.begin(), t.color_ptr.end(), color_ptr);
    if (n_colors_out) *n_colors_out = t.n_colors;
    if (n_levels) *n_levels = t.n_levels;
    if (part_ptr) std::copy(t.part_ptr.begin(), t.part_ptr.end(), part_ptr);
    if (n_send) for (int p = 0; p < std::max(1, n_parts); ++p) n_send[p] = t.send_ptr[p + 1] - t.send_ptr[p];
    return CWR_OK;
}

// ------------------------------------------------------------------------------------------------
// domain decomposition plumbing: one handle per GPU/process; CUDA IPC maps every rank's slab into every peer
// ------------------------------------------------------------------------------------------------
int cwr_dd_export(cwr_handle* h, void* ipc_handle) {
    if (!h || !ipc_handle) return CWR_EINVAL;
    CK(cudaSetDevice(h->device));
    cudaIpcMemHandle_t mh;
    CK(cudaIpcGetMemHandle(&mh, h->d_slab));
    static_assert(sizeof(mh) == CWR_IPC_HANDLE_BYTES, "cudaIpcMemHandle_t size");
    std::memcpy(ipc_handle, &mh, sizeof mh);
    return CWR_OK;
}

int cwr_dd_attach(cwr_handle* h, const void* ipc_handles) {
    if (!h) return CWR_EINVAL;
    if (h->world == 1) { h->attached = true; return CWR_OK; }
    if (!ipc_handles) FAIL(CWR_EINVAL, "NULL handles");
    if (h->attached) FAIL(CWR_EINVAL, "already attached");
    CK(cudaSetDevice(h->device));
    for (int q = 0; q < h->world; ++q) {
        if (q == h->rank) continue;
        cudaIpcMemHandle_t mh;
        std::memcpy(&mh, (const char*)ipc_handles + (size_t)q * CWR_IPC_HANDLE_BYTES, sizeof mh);
        void* p = nullptr;
        CK(cudaIpcOpenMemHandle(&p, mh, cudaIpcMemLazyEnablePeerAccess));
        h->peer_maps.push_back(p);
        h->M.peer_base[q] = (char*)p;
    }
    h->attached = true;
    h->hint_done = true;       // ownership is now shared knowledge: no recolouring after this point
    return CWR_OK;
}

int cwr_dd_layout(cwr_handle* h, cwr_dd_info* out, uint8_t* owned_cells, uint8_t* owned_edges) {
    if (!h) return CWR_EINVAL;
    const Topology& tp = h->topo;
    const DeviceModel& M = h->M;
    if (out) {
        out->rank = h->rank; out->world = h->world;
        out->rows_owned = M.row_hi - M.row_lo;
        out->rows_sent = tp.send_ptr[h->rank + 1] - tp.send_ptr[h->rank];
        out->neighbour_mask = (int)M.nbr_mask;
        out->n_colors = tp.n_colors; out->n_levels = tp.n_levels;
    }
    if (owned_cells) for (int i = 0; i < h->n; ++i) { const int32_t r = tp.new_of_old[i]; owned_cells[i] = r >= M.row_lo && r < M.row_hi; }
    if (owned_edges) {
        std::fill(owned_edges, owned_edges + h->E, (uint8_t)0);
        for (int ep = M.ie_lo; ep < M.ie_hi; ++ep) owned_edges[tp.eperm[ep]] = 1;
        for (int g = M.ge_lo; g < M.ge_hi; ++g) owned_edges[tp.eperm[tp.E_int + g]] = 1;
    }
    return CWR_OK;
}

int cwr_strip_layout(int n_real, int n_face, int n_edge, const int32_t* f1, const int32_t* f2, int n_colors, const float* flow_hint,
                     int n_parts, int n_strips, int* n_colors_out, int* nbr_total, int32_t* new_of_old, int32_t* strip_cptr,
                     int32_t* strip_nptr, int32_t* strip_nbr, uint8_t* color_of, int strip_cap) {
    if (!f1 || !f2) return CWR_EINVAL;
    Topology t;
    const std::string terr = build_topology(n_real, n_face, n_edge, f1, f2, true, n_colors, flow_hint, std::max(1, n_parts), t, n_strips,
                                            std::max(0, strip_cap));
    if (!terr.empty()) { g_create_error = terr; return CWR_EINVAL; }
    if (n_colors_out) *n_colors_out = t.n_colors;
    if (nbr_total) *nbr_total = (int)t.strip_nbr.size();
    if (new_of_old) std::copy(t.new_of_old.begin(), t.new_of_old.end(), new_of_old);
    if (strip_cptr) std::copy(t.strip_cptr.begin(), t.strip_cptr.end(), strip_cptr);
    if (strip_nptr) std::copy(t.strip_nptr.begin(), t.strip_nptr.end(), strip_nptr);
    if (strip_nbr) std::copy(t.strip_nbr.begin(), t.strip_nbr.end(), strip_nbr);
    if (color_of) std::copy(t.color_of.begin(), t.color_of.end(), color_of);
    return CWR_OK;
}

int cwr_get_options(const cwr_handle* h, cwr_options* out) {
    if (!h || !out) return CWR_EINVAL;
    *out = h->opt;
    out->precond_colors = (h->gauss_seidel || h->tiny) ? h->topo.n_colors : 0;
    out->precond_sweep = (h->gauss_seidel || h->tiny) ? 1 : 0;
    out->solver_path = h->tiny ? (h->chip_ns > 0 ? 4 : 3) : (h->small_path ? 2 : 1);
    out->solver = h->dc ? 2 : 1;
    out->precond_sync = h->gauss_seidel ? (h->tma ? 4 : (h->pipelined ? 3 : (h->strips ? 2 : 1))) : 0;
    return CWR_OK;
}

int cwr_stream(cwr_handle* h, void** s) {
    if (!h || !s) return CWR_EINVAL;
    *s = (void*)h->stream;
    return CWR_OK;
}

int cwr_counters(cwr_handle* h, int64_t* launches, int64_t* iterations) {
    if (!h) return CWR_EINVAL;
    if (launches) *launches = h->launches;
    if (iterations) *iterations = h->iterations;
    return CWR_OK;
}

int cwr_solver_stats(cwr_handle* h, int64_t* sweeps, int64_t* fallbacks, int* n_strips, int* max_strip_neighbours) {
    if (!h) return CWR_EINVAL;
    if (sweeps) *sweeps = h->sweeps_total;
    if (fallbacks) *fallbacks = h->fallbacks;
    if (n_strips) *n_strips = h->strips ? h->n_strips : 0;
    if (max_strip_neighbours) *max_strip_neighbours = h->strips ? h->topo.max_strip_nbr : 0;
    return CWR_OK;
}

int cwr_profile(cwr_handle* h, int enable, double* ms, int64_t* counts) {
    if (!h) return CWR_EINVAL;
    if (ms) std::copy(h->fam_ms, h->fam_ms + CWR_PROFILE_FAMILIES, ms);
    if (counts) std::copy(h->fam_count, h->fam_count + CWR_PROFILE_FAMILIES, counts);
    if (enable >= 0) {
        if ((enable != 0) != h->profiling) {
            std::fill(h->fam_ms, h->fam_ms + CWR_PROFILE_FAMILIES, 0.0);
            std::fill(h->fam_count, h->fam_count + CWR_PROFILE_FAMILIES, (int64_t)0);
        }
        h->profiling = enable != 0;
        h->ev_used = 0;
    }
    return CWR_OK;
}

int cwr_time_spmm(cwr_handle* h, int reps, double* ms_per_launch, double* algorithmic_bytes) {
    if (!h) return CWR_EINVAL;
    if (reps <= 0) FAIL(CWR_EINVAL, "reps must be positive");
    if (h->lhs_step < 0) FAIL(CWR_EINVAL, "assemble a LHS (take a step) before timing the product");
    CK(cudaSetDevice(h->device));
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    DeviceModel& M = h->M;
    // x = p (left by the last solve), y = v ; both are scratch between steps
    for (int w = 0; w < 3; ++w) { KC_DISPATCH(h->KC, (k_spmm<KC, VEC, MODE_PLAIN, double><<<h->grid_spmm, kThreads, 0, h->stream>>>(M, M.p, M.v))); }
    CK(cudaEventRecord(e0, h->stream));
    for (int r = 0; r < reps; ++r) { KC_DISPATCH(h->KC, (k_spmm<KC, VEC, MODE_PLAIN, double><<<h->grid_spmm, kThreads, 0, h->stream>>>(M, M.p, M.v))); }
    CK(cudaEventRecord(e1, h->stream));
    CK(cudaEventSynchronize(e1));
    h->launches += reps + 3;
    float ms = 0.f;
    CK(cudaEventElapsedTime(&ms, e0, e1));
    CK(cudaEventDestroy(e0)); CK(cudaEventDestroy(e1));
    if (ms_per_launch) *ms_per_launch = (double)ms / reps;
    if (algorithmic_bytes)
        *algorithmic_bytes = 12.0 * (double)h->topo.nnz + 4.0 * (h->n + 1.0) + 16.0 * (double)h->n * h->K;   /* SURVEY 8d */
    return CWR_OK;
}

}  // extern "C"
