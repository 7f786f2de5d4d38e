// raftk.cu -- sm_100a kernels + C ABI for the RAO-solve hot path (see include/raftk.h, DESIGN.md).
//
// Kernels
//   k_depth_table   : depth-decay functions cosh/sinh ratios per (node, frequency)      helpers.py:207-222
//   k_excitation    : sea state -> zeta, node phase table, strip inertial + BEM excitation
//                     raft_fowt.py:1732-1888, raft_member.py:1899-1992, helpers.py:188-236,703-760
//   k_drag_solve    : per (design, case) CTA cluster: drag linearisation (cross-frequency RMS),
//                     B_drag, F_drag, impedance assembly, 6x6 complex LU per frequency, convergence,
//                     relaxation          raft_model.py:1052-1142, raft_fowt.py:1891-1957,
//                                         raft_member.py:1995-2152, helpers.py:149-184,678-684
//   k_system_solve  : dense n x n complex solve per frequency (farm)      raft_model.py:1164-1216
//   k_fp64_peak     : DFMA micro-benchmark for the FP64 roofline denominator
//
// Algebra used by the kernels (DESIGN.md section 4): with member frame (q,p1,p2), node position
// r_j = rA + ls_j q and lever arm a = rA - r_ref, a 3-vector d in {q,p1,p2} at node j acts on the
// 6-DOF body through V_jd = [d ; r_j x d]:
//     V_jq = [q ; a x q],  V_jp1 = [p1 ; a x p1 + ls_j p2],  V_jp2 = [p2 ; a x p2 - ls_j p1]
// (q x p1 = p2, q x p2 = -p1).  Wave velocity projections are c_jd(w) = zeta w E_j (C_j h_d + i S_j d_z)
// with E_j = exp(-i k (x_j cos b + y_j sin b)), h_d = d_x cos b + d_y sin b, and (C_j,S_j) the depth
// functions.  Everything the reference does per (node, frequency) with 3x3 / 6x6 matrices reduces to
// complex scalars per node and a handful of sums per member.
#include <cuda_runtime.h>
#include <cooperative_groups.h>
#include <math_constants.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <mutex>
#include <algorithm>
#include <type_traits>
#include <vector>

#include "../../include/raftk.h"

namespace cg = cooperative_groups;

// ------------------------------------------------------------------------------------------------
// error handling
// ------------------------------------------------------------------------------------------------
static thread_local char g_err[512] = "";
static long long g_launches = 0;

static int set_err(int code, const char *fmt, const char *a = "", const char *b = "")
{
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return code;
}
#define CUDA_TRY(expr)                                                                          \
    do {                                                                                        \
        cudaError_t _e = (expr);                                                                \
        if (_e != cudaSuccess) return set_err(RAFTK_ECUDA, "%s: %s", #expr, cudaGetErrorString(_e)); \
    } while (0)

// ---- per-device opt-in for > 48 KB of dynamic shared memory ------------------------------------------
// cudaFuncSetAttribute applies to the CURRENT device only, so the high-water mark is kept per device
// (a process may drive several GPUs through DeviceSession(device=...)).
#define RAFTK_MAX_DEV 64
static int cur_dev()
{
    int d = 0;
    if (cudaGetDevice(&d) != cudaSuccess) { cudaGetLastError(); return 0; }
    return (d >= 0 && d < RAFTK_MAX_DEV) ? d : 0;
}
struct SmemOptIn {
    std::mutex mu;
    size_t set[RAFTK_MAX_DEV];
    explicit SmemOptIn(size_t floor = 0) { for (auto &v : set) v = floor; }
    template <class K> cudaError_t ensure(K kernel, size_t bytes)
    {
        std::lock_guard<std::mutex> lk(mu);
        const int d = cur_dev();
        if (bytes <= set[d]) return cudaSuccess;
        cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        if (e == cudaSuccess) set[d] = bytes;
        return e;
    }
};

// ---- optional per-kernel event timing (roofline report) ----------------------------------------------
struct ProfRec { cudaEvent_t a, b; int kind; };
static bool g_prof_on = false;
static std::vector<ProfRec> g_prof;
static std::mutex g_prof_mu;

static void prof_begin_call()
{
    if (!g_prof_on) return;
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (auto &r : g_prof) { cudaEventDestroy(r.a); cudaEventDestroy(r.b); }
    g_prof.clear();
}
struct ProfScope {
    cudaStream_t st; int idx = -1;
    ProfScope(cudaStream_t s, int kind) : st(s)
    {
        if (!g_prof_on) return;
        std::lock_guard<std::mutex> lk(g_prof_mu);
        ProfRec r; r.kind = kind;
        cudaEventCreate(&r.a); cudaEventCreate(&r.b);
        cudaEventRecord(r.a, st);
        g_prof.push_back(r); idx = (int)g_prof.size() - 1;
    }
    ~ProfScope()
    {
        if (idx < 0) return;
        std::lock_guard<std::mutex> lk(g_prof_mu);
        cudaEventRecord(g_prof[idx].b, st);
    }
};
extern "C" void raftk_profile_enable(int on) { g_prof_on = on != 0; }
extern "C" int raftk_profile_read(double ms[3], int launches[3])
{
    std::lock_guard<std::mutex> lk(g_prof_mu);
    for (int t = 0; t < 3; t++) { ms[t] = 0.0; launches[t] = 0; }
    for (auto &r : g_prof) {
        if (cudaEventSynchronize(r.b) != cudaSuccess) return RAFTK_ECUDA;
        float f = 0.f;
        if (cudaEventElapsedTime(&f, r.a, r.b) != cudaSuccess) return RAFTK_ECUDA;
        ms[r.kind] += f; launches[r.kind]++;
    }
    return RAFTK_OK;
}

extern "C" int raftk_version(void) { return RAFTK_VERSION; }
extern "C" const char *raftk_last_error(void) { return g_err; }
extern "C" long long raftk_launch_count(void) { return g_launches; }

#include "raftk_common.cuh"
#include "raftk_tables.cuh"
#include "raftk_fused.cuh"
#include "raftk_fused2.cuh"
#include "raftk_qtf.cuh"
#include "raftk_slender.cuh"
#include "raftk_general.cuh"
#include "raftk_misc.cuh"
#include "raftk_builder.h"

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static DesignsDev to_dev(const raftk_designs *d, int max_nodes, int max_members)
{
    DesignsDev D;
    D.nD = d->n_designs; D.nw = d->nw; D.max_nodes = max_nodes; D.max_members = max_members; D.n_bem_head = d->n_bem_head;
    D.depth = d->depth; D.rho = d->rho; D.g = d->g; D.dw = d->dw;
    D.w = d->w; D.k = d->k; D.member_offset = d->member_offset;
    D.mem_frame = d->mem_frame; D.mem_rA = d->mem_rA; D.mem_arm = d->mem_arm;
    D.mem_node_start = d->mem_node_start; D.mem_circ = d->mem_circ;
    D.node_ls = d->node_ls; D.node_cd_q = d->node_cd_q; D.node_cd_p1 = d->node_cd_p1; D.node_cd_p2 = d->node_cd_p2;
    D.node_in_q = d->node_in_q; D.node_in_p1 = d->node_in_p1; D.node_in_p2 = d->node_in_p2; D.node_pa = d->node_pa;
    D.node_in_p1_w = reinterpret_cast<const double2 *>(d->node_in_p1_w);
    D.node_in_p2_w = reinterpret_cast<const double2 *>(d->node_in_p2_w);
    D.M0 = d->M0; D.B0 = d->B0; D.C0 = d->C0; D.A_w = d->A_w; D.B_w = d->B_w;
    D.bem_headings = d->bem_headings; D.X_BEM = d->X_BEM; D.bem_xyh = d->bem_xyh;
    return D;
}

static CasesDev to_dev(const raftk_cases *c)
{
    CasesDev C;
    C.nC = c->n_cases; C.Hs = c->Hs; C.Tp = c->Tp; C.gamma = c->gamma; C.beta_deg = c->beta_deg;
    C.zeta_in = c->zeta; C.spec = c->spec; C.primary = c->primary; C.F_2nd = c->F_2nd;
    return C;
}

static size_t align_up(size_t x, size_t a) { return (x + a - 1) / a * a; }

static size_t chunk_bytes(int nDc, int nC, int max_nodes, int nw)
{
    size_t b = 0;
    b += align_up((size_t)nDc * max_nodes * nw * sizeof(double2), 256);
    b += align_up((size_t)nDc * nC * max_nodes * nw * sizeof(double2), 256);
    b += align_up((size_t)nDc * nC * 6 * nw * sizeof(double2), 256);
    b += align_up((size_t)nC * nw * sizeof(double), 256);
    return b;
}

extern "C" size_t raftk_workspace_bytes(const raftk_designs *d, int32_t n_cases)
{
    if (!d || d->n_designs <= 0) return 0;
    const size_t cap = (size_t)8 << 30;       // plan at most 8 GiB; larger batches run in design chunks
    const int maxn = d->max_nodes > 0 ? d->max_nodes : 1;
    const size_t full = chunk_bytes(d->n_designs, n_cases, maxn, d->nw);
    const size_t one = chunk_bytes(1, n_cases, maxn, d->nw);
    return full <= cap ? full : std::max(cap, one);
}

struct FPlan { int CS, nwl, T, nchunk, maxW, maxH, maxZ; size_t smem; bool f0_global; };
static bool fused_plan(const raftk_designs *d, int units, int requested_cs, bool have_ws, FPlan &pl);

static int validate(const raftk_designs *d, const raftk_cases *c)
{
    if (!d || !c) return set_err(RAFTK_EINVAL, "null designs/cases");
    if (d->n_designs <= 0 || d->nw <= 0 || c->n_cases <= 0) return set_err(RAFTK_EINVAL, "empty batch (n_designs, nw, n_cases must be > 0)");
    if (d->max_nodes <= 0 || d->max_members <= 0) return set_err(RAFTK_EINVAL, "max_nodes/max_members must be > 0");
    if (d->max_members > 512 || d->max_nodes > 4096) return set_err(RAFTK_EINVAL, "design too large for the shared-memory tables");
    if ((d->node_in_p1_w == nullptr) != (d->node_in_p2_w == nullptr)) return set_err(RAFTK_EINVAL, "node_in_p1_w / node_in_p2_w must both be given or both NULL");
    return 0;
}

// ---- second-order forces from the designs' QTF table -------------------------------------------------
static int validate_qtf(const raftk_designs *d, const raftk_cases *c)
{
    if (!d || !c) return set_err(RAFTK_EINVAL, "null designs/cases");
    if (d->n_designs <= 0 || d->nw <= 0 || c->n_cases <= 0) return set_err(RAFTK_EINVAL, "empty batch (n_designs, nw, n_cases must be > 0)");
    if (d->n_qtf_w < 2 || d->n_qtf_head < 1 || !d->qtf || !d->qtf_w || !d->qtf_heads)
        return set_err(RAFTK_EINVAL, "designs carry no QTF table (n_qtf_w >= 2, n_qtf_head >= 1, qtf, qtf_w, qtf_heads)");
    if (d->qtf_shared < 0 || d->qtf_shared > 2) return set_err(RAFTK_EINVAL, "qtf_shared must be 0, 1 or 2");
    if ((size_t)d->nw * 20 > 227 * 1024) return set_err(RAFTK_EINVAL, "nw too large for the second-order force kernel's shared-memory tables");
    return 0;
}

static int run_qtf(const raftk_designs *d, const raftk_cases *c, double *F2, double *F2mean, cudaStream_t st)
{
    int rc = validate_qtf(d, c);
    if (rc) return rc;
    if (!F2) return set_err(RAFTK_EINVAL, "second-order force needs the F_2nd buffer");
    CasesDev C = to_dev(c);
    QtfParams P;
    P.nD = d->n_designs; P.shared = d->qtf_shared;
    P.n2 = d->n_qtf_w; P.nh = d->n_qtf_head; P.nw = d->nw; P.dw = d->dw;
    P.w = d->w; P.qw = d->qtf_w; P.qh = d->qtf_heads;
    P.qtf = reinterpret_cast<const double2 *>(d->qtf);
    P.F2 = F2; P.F2mean = F2mean;
    const size_t smem = (size_t)d->nw * 20;
    static SmemOptIn opt_plain(48 * 1024), opt_mix(48 * 1024), opt_tiles(48 * 1024);
    CUDA_TRY(opt_plain.ensure(k_qtf_force<false>, smem));
    CUDA_TRY(opt_mix.ensure(k_qtf_force<true>, smem));
    if (P.shared != 1 && d->n_designs > 65535) return set_err(RAFTK_EINVAL, "second-order force: more than 65535 designs per call");
    if (c->n_cases > 65535) return set_err(RAFTK_EINVAL, "second-order force: more than 65535 cases per call");
    // tile variant (registers hold the table-cell corners, systolic diagonal accumulators) when its shared-memory
    // tables fit and the frequency rows fit k_qtf_finish's register staging; RAFTK_QTF_DIAG=1 forces the diagonal kernel
    const int ncell = d->n_qtf_w - 1;
    const size_t tsmem = (size_t)d->nw * 68 + (size_t)ncell * 8 + 16;
    const bool tiles = !getenv("RAFTK_QTF_DIAG") && tsmem <= 226 * 1024 && d->nw <= 4096;
    if (tiles) {
        CUDA_TRY(opt_tiles.ensure(k_qtf_tiles, tsmem));
        QtfTileParams TP;
        TP.q = P; TP.ncell = ncell;
        const size_t rows = (size_t)((P.shared == 1) ? 1 : d->n_designs) * c->n_cases * 6 * d->nw;
        CUDA_TRY(cudaMemsetAsync(F2, 0, rows * sizeof(double), st));
        dim3 gt(QT_GROUPS, c->n_cases, P.shared == 1 ? 1 : d->n_designs);
        k_qtf_tiles<<<gt, QT_THREADS, tsmem, st>>>(C, TP);
        dim3 gf(6, c->n_cases, P.shared == 1 ? 1 : d->n_designs);
        k_qtf_finish<<<gf, 256, 0, st>>>(C, P);
        g_launches += 2;
        CUDA_TRY(cudaGetLastError());
        return RAFTK_OK;
    }
    const int ntasks = d->nw / 2 + 1, per_cta = (QTF_THREADS / 32) * QTF_TASKS_PER_WARP;
    dim3 grid((ntasks + per_cta - 1) / per_cta, c->n_cases, P.shared == 1 ? 1 : d->n_designs);
    if (P.nh > 1) k_qtf_force<true><<<grid, QTF_THREADS, smem, st>>>(C, P);
    else k_qtf_force<false><<<grid, QTF_THREADS, smem, st>>>(C, P);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return RAFTK_OK;
}

extern "C" int raftk_second_order_force_dev(const raftk_designs *d, const raftk_cases *c, const raftk_outputs *out, void *stream)
{
    if (!out || !out->F_2nd) return set_err(RAFTK_EINVAL, "outputs.F_2nd is required");
    return run_qtf(d, c, out->F_2nd, out->F_2nd_mean, (cudaStream_t)stream);
}

static int pick_cluster(int units, int nw, int requested)
{
    if (requested == 1 || requested == 2 || requested == 4 || requested == 8) {
        int cs = requested;
        while (cs > 1 && nw / cs < 32) cs >>= 1;
        return cs;
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    int cs = 1;
    // fill ~2 CTAs per SM, keep >= 128 frequencies per CTA, and keep 12*nwl doubles of state <= 48 KB
    while (cs < 8 && (units * cs < 2 * sms || nw / cs > 512) && nw / (cs * 2) >= 128) cs <<= 1;
    return cs;
}

struct Plan { int CS, nwl, nchunk; size_t smem; };

static int make_plan(const raftk_designs *d, int units_hint, int requested_cs, Plan &pl)
{
    pl.CS = pick_cluster(units_hint, d->nw, requested_cs);
    pl.nwl = (d->nw + pl.CS - 1) / pl.CS;
    pl.nchunk = (d->max_nodes + CHUNK_NODES - 1) / CHUNK_NODES;
    pl.smem = smem_doubles(d->max_members, d->max_nodes, pl.nchunk, SOLVE_THREADS / 32, pl.nwl) * sizeof(double)
              + (size_t)d->max_members * 3 * sizeof(int) + 16;
    if (pl.smem > 227 * 1024) return set_err(RAFTK_EINVAL, "shared-memory plan exceeds 227 KB (nw per CTA too large)");
    return 0;
}

// ---- fused (v2) planner / launcher -----------------------------------------------------------------

static bool fused_try(const raftk_designs *d, int cs, bool have_ws, FPlan &pl)
{
    pl.CS = cs;
    pl.nwl = (d->nw + cs - 1) / cs;
    pl.T = pl.nwl > 128 ? 256 : 128;
    pl.nchunk = (d->max_nodes + CHUNK_NODES - 1) / CHUNK_NODES;
    pl.maxW = d->max_w_classes > 0 ? d->max_w_classes : d->max_nodes;
    pl.maxH = d->max_h_classes > 0 ? d->max_h_classes : d->max_nodes;
    pl.maxZ = d->max_z_classes > 0 ? std::min(d->max_z_classes, d->max_members) : d->max_members;
    // 255 registers cap residency at 256 threads per SM (measured: 168 registers / 3 CTAs is slower, the LU
    // spills); shared memory must allow 2 CTAs of 128 threads or 1 of 256.  The linear excitation F0 lives in
    // shared memory when it fits, else in the caller's workspace.
    const size_t limit = (pl.T == 128) ? (size_t)112 * 1024 : (size_t)226 * 1024;
    pl.f0_global = false;
    pl.smem = fused_smem_bytes(d->max_members, d->max_nodes, pl.nchunk, pl.T / 32, pl.nwl, pl.maxW, pl.maxH, pl.maxZ, true);
    if (pl.smem > limit && have_ws) {
        pl.f0_global = true;
        pl.smem = fused_smem_bytes(d->max_members, d->max_nodes, pl.nchunk, pl.T / 32, pl.nwl, pl.maxW, pl.maxH, pl.maxZ, false);
    }
    return pl.smem <= limit && pl.nwl <= 2 * pl.T;
}

static bool fused_plan(const raftk_designs *d, int units, int requested_cs, bool have_ws, FPlan &pl)
{
    if (getenv("RAFTK_FORCE_V1")) return false;
    if (requested_cs == 1 || requested_cs == 2 || requested_cs == 4 || requested_cs == 8) {
        int cs = requested_cs;
        while (cs > 1 && d->nw / cs < 32) cs >>= 1;
        return fused_try(d, cs, have_ws, pl);
    }
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    FPlan best; bool have = false;
    if (units >= 4 * sms) {                       // plenty of units: smallest cluster whose slice fits on chip
        for (int cs = 1; cs <= 8 && !have; cs <<= 1) { FPlan t; if (fused_try(d, cs, have_ws, t) && t.nwl <= t.T) { best = t; have = true; } }
        for (int cs = 1; cs <= 8 && !have; cs <<= 1) { FPlan t; if (fused_try(d, cs, have_ws, t)) { best = t; have = true; } }
    } else {                                      // few units: largest cluster that keeps >= 128 bins per CTA
        for (int cs = 8; cs >= 1 && !have; cs >>= 1) {
            if (cs > 1 && d->nw / cs < 128) continue;
            FPlan t; if (fused_try(d, cs, have_ws, t)) { best = t; have = true; }
        }
    }
    if (have) pl = best;
    return have;
}

template <int T>
static int fused_launch(const DesignsDev &D, const CasesDev &C, const FusedParams &P, const FPlan &pl, int units, cudaStream_t st)
{
    static SmemOptIn opt;
    CUDA_TRY(opt.ensure(k_rao_fused<T>, pl.smem));
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)((size_t)units * pl.CS), 1, 1);
    cfg.blockDim = dim3(T, 1, 1);
    cfg.dynamicSmemBytes = pl.smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = pl.CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    {
        ProfScope ps(st, 2);
        CUDA_TRY(cudaLaunchKernelEx(&cfg, k_rao_fused<T>, D, C, P));
    }
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return RAFTK_OK;
}

static int run_fused(const raftk_designs *d, const raftk_cases *c, const raftk_solve_opts *o, const raftk_outputs *out,
                     const FPlan &pl, void *workspace, size_t wbytes, cudaStream_t st, const raftk_peers *peers = nullptr)
{
    prof_begin_call();
    DesignsDev D = to_dev(d, d->max_nodes, d->max_members);
    CasesDev C = to_dev(c);
    FusedParams P;
    P.n_iter = o->n_iter; P.CS = pl.CS; P.nwl = pl.nwl; P.maxW = pl.maxW; P.maxH = pl.maxH; P.maxZ = pl.maxZ;
    P.tol = o->tol; P.xi_start = o->xi_start;
    P.Xi_out = reinterpret_cast<double2 *>(out->Xi);
    P.Fdrag_out = reinterpret_cast<double2 *>(out->F_drag);
    P.Finer_out = reinterpret_cast<double2 *>(out->F_iner);
    P.Fbem_out = reinterpret_cast<double2 *>(out->F_BEM);
    P.Bdrag_out = out->B_drag; P.zeta_out = out->zeta; P.status = out->status;
    P.Xilast_out = reinterpret_cast<double2 *>(out->Xi_last);
    P.Xi_init = reinterpret_cast<const double2 *>(c->Xi_init);
    P.F0g = pl.f0_global ? reinterpret_cast<double2 *>(workspace) : nullptr;
    const int units = d->n_designs * c->n_cases;
    P.lin_g = nullptr; P.phase = -1;
    P.n_peers = 0; P.peer_rank = 0;
    for (int p = 0; p < RAFTK_MAX_PEERS; p++) { P.peer_Xi[p] = nullptr; P.peer_status[p] = nullptr; }
    if (peers && peers->n_ranks > 1) {
        P.n_peers = peers->n_ranks; P.peer_rank = peers->rank;
        const size_t units_per_rank = peers->block_elems / ((size_t)6 * d->nw);
        for (int p = 0; p < peers->n_ranks; p++) {
            P.peer_Xi[p] = reinterpret_cast<double2 *>(peers->gathered[p]) + (size_t)peers->rank * peers->block_elems;
            P.peer_status[p] = peers->status[p] ? peers->status[p] + (size_t)peers->rank * units_per_rank * 4 : nullptr;
        }
    }
    if (c->primary) {                                  // wave trains: primaries first, then the trains that follow them
        const size_t f0b = align_up((size_t)units * 6 * d->nw * sizeof(double2), 256);
        const size_t need = f0b + (size_t)units * ((size_t)NCOEF * d->max_nodes + 36) * sizeof(double);
        if (!workspace || wbytes < need) return set_err(RAFTK_ENOMEM, "wave-train cases need raftk_solve_workspace_bytes() of workspace");
        P.lin_g = reinterpret_cast<double *>(static_cast<char *>(workspace) + f0b);
        for (int phase = 0; phase < 2; phase++) {
            P.phase = phase;
            const int rc = (pl.T == 128) ? fused_launch<128>(D, C, P, pl, units, st) : fused_launch<256>(D, C, P, pl, units, st);
            if (rc) return rc;
        }
        return RAFTK_OK;
    }
    if (pl.T == 128) return fused_launch<128>(D, C, P, pl, units, st);
    return fused_launch<256>(D, C, P, pl, units, st);
}

// ---- fused2 (two bins per thread, TMA-staged plan blob) planner / launcher --------------------------------------------
struct F2Plan { int CS, nwl, nchunk, maxW, maxH, maxZ; size_t smem, blob, o_lin, o_E, o_A, o_plan, ws_bytes; };

static bool fused2_plan(const raftk_designs *d, int n_cases, int requested_cs, F2Plan &pl)
{
    if (getenv("RAFTK_FORCE_V1") || getenv("RAFTK_FUSED_GEN1")) return false;      // A/B: first-generation fused kernel
    if (d->max_nodes <= 0 || d->max_members <= 0) return false;
    int cs;
    if (requested_cs == 1 || requested_cs == 2 || requested_cs == 4 || requested_cs == 8) cs = requested_cs;
    else { cs = 1; while (cs < 8 && (d->nw + cs - 1) / cs > 2 * F2_T) cs <<= 1; }
    pl.CS = cs;
    pl.nwl = (d->nw + cs - 1) / cs;
    // two bins per thread pay when most threads own two: 192 < bins per CTA <= 256; otherwise the one-bin kernel runs
    if (pl.nwl > 2 * F2_T || pl.nwl <= (3 * F2_T) / 2) return false;
    pl.nchunk = (d->max_nodes + CHUNK_NODES - 1) / CHUNK_NODES;
    pl.maxW = d->max_w_classes > 0 ? d->max_w_classes : d->max_nodes;
    pl.maxH = d->max_h_classes > 0 ? d->max_h_classes : d->max_nodes;
    pl.maxZ = d->max_z_classes > 0 ? std::min(d->max_z_classes, d->max_members) : d->max_members;
    pl.smem = fused2_smem_bytes(d->max_members, d->max_nodes, pl.nchunk, pl.nwl, pl.maxW, pl.maxH, pl.maxZ);
    if (pl.smem > (size_t)113 * 1024) return false;                               // two CTAs per SM
    const size_t units = (size_t)d->n_designs * n_cases;
    pl.blob = (size_t)plan_layout(d->max_members, d->max_nodes, pl.maxW, pl.maxH, pl.maxZ).total;
    size_t o = align_up(units * 6 * d->nw * sizeof(double2), 256);                 // F0 (same place as the first-generation kernel)
    pl.o_lin = o; o += align_up(units * ((size_t)NCOEF * d->max_nodes + 36) * sizeof(double), 256);
    pl.o_E = o; o += align_up(units * (size_t)d->max_members * d->nw * sizeof(double2), 256);
    pl.o_A = o; o += align_up(units * (size_t)pl.maxZ * d->nw * sizeof(double2), 256);
    pl.o_plan = o; o += align_up((size_t)d->n_designs * pl.blob * sizeof(double), 256);
    pl.ws_bytes = o;
    return true;
}

static int run_fused2(const raftk_designs *d, const raftk_cases *c, const raftk_solve_opts *o, const raftk_outputs *out,
                      const F2Plan &pl, void *workspace, cudaStream_t st, const raftk_peers *peers)
{
    prof_begin_call();
    DesignsDev D = to_dev(d, d->max_nodes, d->max_members);
    CasesDev C = to_dev(c);
    char *ws = static_cast<char *>(workspace);
    FusedParams P;
    memset(&P, 0, sizeof(P));
    P.n_iter = o->n_iter; P.CS = pl.CS; P.nwl = pl.nwl; P.maxW = pl.maxW; P.maxH = pl.maxH; P.maxZ = pl.maxZ;
    P.tol = o->tol; P.xi_start = o->xi_start;
    P.Xi_out = reinterpret_cast<double2 *>(out->Xi);
    P.Fdrag_out = reinterpret_cast<double2 *>(out->F_drag);
    P.Finer_out = reinterpret_cast<double2 *>(out->F_iner);
    P.Fbem_out = reinterpret_cast<double2 *>(out->F_BEM);
    P.Bdrag_out = out->B_drag; P.zeta_out = out->zeta; P.status = out->status;
    P.Xilast_out = reinterpret_cast<double2 *>(out->Xi_last);
    P.Xi_init = reinterpret_cast<const double2 *>(c->Xi_init);
    P.F0g = reinterpret_cast<double2 *>(ws);
    P.lin_g = nullptr; P.phase = -1;
    P.Eg = reinterpret_cast<double2 *>(ws + pl.o_E);
    P.Ag = reinterpret_cast<double2 *>(ws + pl.o_A);
    double *plan = reinterpret_cast<double *>(ws + pl.o_plan);
    P.plan = plan; P.plan_stride = pl.blob;
    if (peers && peers->n_ranks > 1) {
        P.n_peers = peers->n_ranks; P.peer_rank = peers->rank;
        const size_t units_per_rank = peers->block_elems / ((size_t)6 * d->nw);
        for (int p = 0; p < peers->n_ranks; p++) {
            P.peer_Xi[p] = reinterpret_cast<double2 *>(peers->gathered[p]) + (size_t)peers->rank * peers->block_elems;
            P.peer_status[p] = peers->status[p] ? peers->status[p] + (size_t)peers->rank * units_per_rank * 4 : nullptr;
        }
    }
    if (!(o->flags & RAFTK_SOLVE_REUSE_PLAN)) {
        ProfScope ps(st, 0);
        const size_t psm = (3 * (size_t)d->max_nodes + d->max_members) * sizeof(double) + (2 * (size_t)d->max_nodes + 2 * d->max_members) * sizeof(int);
        k_fused_plan<<<d->n_designs, 128, psm, st>>>(D, plan, pl.blob, pl.maxW, pl.maxH, pl.maxZ, pl.nwl);
        g_launches++;
    }
    // the lean instantiation unless the call needs a path it compiles out (see k_rao_fused2)
    const bool full = d->A_w || d->B_w || out->F_drag || out->Xi_last || c->primary;
    auto kern = full ? k_rao_fused2<true> : k_rao_fused2<false>;
    static SmemOptIn opt_full, opt_lean;
    CUDA_TRY((full ? opt_full : opt_lean).ensure(kern, pl.smem));
    const int units = d->n_designs * c->n_cases;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)((size_t)units * pl.CS), 1, 1);
    cfg.blockDim = dim3(F2_T, 1, 1);
    cfg.dynamicSmemBytes = pl.smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = pl.CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    const int nphase = c->primary ? 2 : 1;
    if (c->primary) P.lin_g = reinterpret_cast<double *>(ws + pl.o_lin);
    for (int phase = 0; phase < nphase; phase++) {
        P.phase = c->primary ? phase : -1;
        {
            ProfScope ps(st, 2);
            CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, D, C, P));
        }
        g_launches++;
    }
    CUDA_TRY(cudaGetLastError());
    return RAFTK_OK;
}

static int run(const raftk_designs *d, const raftk_cases *c, const raftk_solve_opts *o, const raftk_outputs *out,
               const double *Xi_in, int mode /*0 solve, 1 linearise, 2 excitation only*/, bool do_excitation,
               void *workspace, size_t wbytes, cudaStream_t st, const raftk_peers *peers = nullptr)
{
    int rc = validate(d, c);
    if (rc) return rc;
    const int nD = d->n_designs, nC = c->n_cases, nw = d->nw;
    if (mode == 0) {                                   // fused on-chip solver when the slice fits in shared memory
        F2Plan f2;
        if (fused2_plan(d, nC, o ? o->cluster_size : 0, f2) && workspace && wbytes >= f2.ws_bytes)
            return run_fused2(d, c, o, out, f2, workspace, st, peers);
        FPlan fp;
        const bool have_ws = workspace && wbytes >= (size_t)nD * nC * 6 * nw * sizeof(double2);
        if (fused_plan(d, nD * nC, o ? o->cluster_size : 0, have_ws, fp)) return run_fused(d, c, o, out, fp, workspace, wbytes, st, peers);
        if (peers && peers->n_ranks > 1) return set_err(RAFTK_EINVAL, "the fused exchange needs the fused solver; the design's frequency slice does not fit on chip");
        if (c->primary) return set_err(RAFTK_EINVAL, "wave-train cases (cases.primary) need the fused solver; the design's frequency slice does not fit on chip");
        if (c->Xi_init || out->Xi_last) return set_err(RAFTK_EINVAL, "cases.Xi_init / outputs.Xi_last need the fused solver; the design's frequency slice does not fit on chip");
    }
    if (c->primary && mode != 2) return set_err(RAFTK_EINVAL, "cases.primary is only supported by raftk_solve_dynamics_*");
    if (do_excitation) prof_begin_call();
    DesignsDev D = to_dev(d, d->max_nodes, d->max_members);
    CasesDev C = to_dev(c);
    const size_t one = chunk_bytes(1, nC, d->max_nodes, nw);
    if (!workspace || wbytes < one) return set_err(RAFTK_ENOMEM, "workspace smaller than one design's tables");
    int per = nD;
    while (per > 1 && (chunk_bytes(per, nC, d->max_nodes, nw) > wbytes || per > 65535)) per = (per + 1) / 2;
    if (mode == 1 && !do_excitation && per < nD)
        return set_err(RAFTK_ENOMEM, "linearization needs the whole batch's tables resident in the workspace");

    Plan pl;
    if (mode != 2) {
        rc = make_plan(d, std::min(per, nD) * nC, o ? o->cluster_size : 0, pl);
        if (rc) return rc;
        static SmemOptIn opt;
        CUDA_TRY(opt.ensure(k_drag_solve, pl.smem));
    }

    for (int d0 = 0; d0 < nD; d0 += per) {
        const int nDc = std::min(per, nD - d0);
        Work W;
        W.d0 = d0; W.nDc = nDc;
        char *p = static_cast<char *>(workspace);
        W.depth_tab = reinterpret_cast<double2 *>(p); p += align_up((size_t)nDc * d->max_nodes * nw * sizeof(double2), 256);
        W.phase_tab = reinterpret_cast<double2 *>(p); p += align_up((size_t)nDc * nC * d->max_nodes * nw * sizeof(double2), 256);
        W.F0 = reinterpret_cast<double2 *>(p); p += align_up((size_t)nDc * nC * 6 * nw * sizeof(double2), 256);
        W.zeta = reinterpret_cast<double *>(p);

        if (do_excitation) {
            dim3 g0((nw + 127) / 128, nDc, 1);
            {
                ProfScope ps(st, 0);
                k_depth_table<<<g0, 128, 0, st>>>(D, W);
            }
            g_launches++;
            ExcOut EO;
            EO.F_iner = reinterpret_cast<double2 *>(out->F_iner);
            EO.F_BEM = reinterpret_cast<double2 *>(out->F_BEM);
            EO.zeta = out->zeta;
            dim3 g1((nw + 127) / 128, nC, nDc);
            {
                ProfScope ps(st, 1);
                k_excitation<<<g1, 128, 0, st>>>(D, C, W, EO);
            }
            g_launches++;
        }
        if (mode != 2) {
            SolveParams P;
            P.n_iter = o ? o->n_iter : 0; P.CS = pl.CS; P.nwl = pl.nwl; P.mode = mode;
            P.tol = o ? o->tol : 0.01; P.xi_start = o ? o->xi_start : 0.0;
            P.Xi_in = reinterpret_cast<const double2 *>(Xi_in);
            P.Xi_out = reinterpret_cast<double2 *>(out->Xi);
            P.Fdrag_out = reinterpret_cast<double2 *>(out->F_drag);
            P.Bdrag_out = out->B_drag;
            P.status = out->status;
            cudaLaunchConfig_t cfg;
            memset(&cfg, 0, sizeof(cfg));
            cfg.gridDim = dim3((unsigned)(nDc * nC * pl.CS), 1, 1);
            cfg.blockDim = dim3(SOLVE_THREADS, 1, 1);
            cfg.dynamicSmemBytes = pl.smem;
            cfg.stream = st;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = pl.CS; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            {
                ProfScope ps(st, 2);
                CUDA_TRY(cudaLaunchKernelEx(&cfg, k_drag_solve, D, C, W, P));
            }
            g_launches++;
        }
        CUDA_TRY(cudaGetLastError());
    }
    return RAFTK_OK;
}

extern "C" size_t raftk_solve_workspace_bytes(const raftk_designs *d, int32_t n_cases)
{
    if (!d || d->n_designs <= 0 || n_cases <= 0) return 0;
    F2Plan f2;
    if (fused2_plan(d, n_cases, 0, f2)) return f2.ws_bytes;
    FPlan fp;
    if (d->max_nodes > 0 && d->max_members > 0 && fused_plan(d, d->n_designs * n_cases, 0, true, fp))
        return align_up((size_t)d->n_designs * n_cases * 6 * d->nw * sizeof(double2), 256)
               + align_up((size_t)d->n_designs * n_cases * ((size_t)NCOEF * d->max_nodes + 36) * sizeof(double), 256);
    return raftk_workspace_bytes(d, n_cases);
}

extern "C" int raftk_hydro_excitation_dev(const raftk_designs *d, const raftk_cases *c, const raftk_outputs *out,
                                          void *workspace, size_t workspace_bytes, void *stream)
{
    if (!out) return set_err(RAFTK_EINVAL, "null outputs");
    if (d && c && chunk_bytes(d->n_designs, c->n_cases, d->max_nodes, d->nw) > workspace_bytes)
        return set_err(RAFTK_ENOMEM, "excitation needs the whole batch's tables in the workspace");
    return run(d, c, nullptr, out, nullptr, 2, true, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int raftk_hydro_linearization_dev(const raftk_designs *d, const raftk_cases *c, const double *Xi_in,
                                             const raftk_outputs *out, void *workspace, size_t workspace_bytes, void *stream)
{
    if (!out || !Xi_in) return set_err(RAFTK_EINVAL, "null outputs / Xi_in");
    return run(d, c, nullptr, out, Xi_in, 1, false, workspace, workspace_bytes, (cudaStream_t)stream);
}

extern "C" int raftk_solve_dynamics_dev(const raftk_designs *d, const raftk_cases *c, const raftk_solve_opts *o,
                                        const raftk_outputs *out, void *workspace, size_t workspace_bytes, void *stream)
{
    if (!out || !out->Xi || !out->status || !o) return set_err(RAFTK_EINVAL, "Xi, status and opts are required");
    if (d && c && d->n_qtf_w > 0 && !c->F_2nd) {          // potSecOrder 2: the solve computes the force itself (raft_model.py:1035-1038)
        if (!out->F_2nd) return set_err(RAFTK_EINVAL, "designs carry a QTF: pass outputs.F_2nd as the buffer, or cases.F_2nd precomputed");
        int rc = run_qtf(d, c, out->F_2nd, out->F_2nd_mean, (cudaStream_t)stream);
        if (rc) return rc;
        raftk_cases cc = *c;
        cc.F_2nd = out->F_2nd;
        return run(d, &cc, o, out, nullptr, 0, true, workspace, workspace_bytes, (cudaStream_t)stream);
    }
    return run(d, c, o, out, nullptr, 0, true, workspace, workspace_bytes, (cudaStream_t)stream);
}

// ---- multi-GPU exchange fused into the solve (peer stores over NVLink) ------------------------------------------
extern "C" int raftk_peer_alloc(size_t bytes, void **dev_ptr, unsigned char handle[64])
{
    if (!dev_ptr || !handle || bytes == 0) return set_err(RAFTK_EINVAL, "peer_alloc: null argument / zero size");
    void *p = nullptr;
    CUDA_TRY(cudaMalloc(&p, bytes));
    cudaError_t e = cudaMemset(p, 0, bytes);
    cudaIpcMemHandle_t h;
    if (e == cudaSuccess) e = cudaIpcGetMemHandle(&h, p);
    if (e != cudaSuccess) { cudaFree(p); return set_err(RAFTK_ECUDA, "peer_alloc: %s", cudaGetErrorString(e)); }
    static_assert(sizeof(cudaIpcMemHandle_t) == 64, "CUDA IPC handle size");
    memcpy(handle, &h, 64);
    *dev_ptr = p;
    return RAFTK_OK;
}
extern "C" int raftk_peer_free(void *dev_ptr)
{
    if (dev_ptr) CUDA_TRY(cudaFree(dev_ptr));
    return RAFTK_OK;
}
extern "C" int raftk_peer_open(const unsigned char handle[64], void **dev_ptr)
{
    if (!dev_ptr || !handle) return set_err(RAFTK_EINVAL, "peer_open: null argument");
    cudaIpcMemHandle_t h;
    memcpy(&h, handle, 64);
    CUDA_TRY(cudaIpcOpenMemHandle(dev_ptr, h, cudaIpcMemLazyEnablePeerAccess));
    return RAFTK_OK;
}
extern "C" int raftk_peer_close(void *dev_ptr)
{
    if (dev_ptr) CUDA_TRY(cudaIpcCloseMemHandle(dev_ptr));
    return RAFTK_OK;
}

static int validate_peers(const raftk_peers *p)
{
    if (!p) return set_err(RAFTK_EINVAL, "null peers");
    if (p->n_ranks < 1 || p->n_ranks > RAFTK_MAX_PEERS || p->rank < 0 || p->rank >= p->n_ranks)
        return set_err(RAFTK_EINVAL, "peers: 1 <= n_ranks <= RAFTK_MAX_PEERS and 0 <= rank < n_ranks");
    for (int r = 0; r < p->n_ranks; r++)
        if (!p->gathered[r] || !p->flags[r]) return set_err(RAFTK_EINVAL, "peers: gathered / flags pointer missing for a rank");
    return 0;
}

extern "C" int raftk_solve_dynamics_gather_dev(const raftk_designs *d, const raftk_cases *c, const raftk_solve_opts *o,
                                               const raftk_outputs *out, const raftk_peers *peers, void *workspace,
                                               size_t workspace_bytes, void *stream)
{
    if (!out || !out->Xi || !out->status || !o) return set_err(RAFTK_EINVAL, "Xi, status and opts are required");
    int rc = validate_peers(peers);
    if (rc) return rc;
    if (!d || !c) return set_err(RAFTK_EINVAL, "null designs/cases");
    if ((size_t)d->n_designs * c->n_cases * 6 * d->nw > peers->block_elems)
        return set_err(RAFTK_EINVAL, "peers.block_elems is smaller than this rank's response block");
    if (out->Xi != peers->gathered[peers->rank] + 2 * (size_t)peers->rank * peers->block_elems)
        return set_err(RAFTK_EINVAL, "outputs.Xi must be this rank's block of its own gathered array");
    if (d->n_qtf_w > 0 && !c->F_2nd) return set_err(RAFTK_EINVAL, "gather solve: pass cases.F_2nd precomputed (raftk_second_order_force_dev)");
    return run(d, c, o, out, nullptr, 0, true, workspace, workspace_bytes, (cudaStream_t)stream, peers);
}

extern "C" int raftk_peer_barrier_dev(const raftk_peers *peers, int32_t *timeout_flag, void *stream)
{
    int rc = validate_peers(peers);
    if (rc) return rc;
    if (peers->epoch == 0) return set_err(RAFTK_EINVAL, "peers.epoch must be > 0");
    PeerFlags F;
    F.n = peers->n_ranks; F.rank = peers->rank; F.epoch = peers->epoch;
    for (int p = 0; p < RAFTK_MAX_PEERS; p++) F.flags[p] = p < peers->n_ranks ? peers->flags[p] : nullptr;
    k_peer_barrier<<<1, 32, 0, (cudaStream_t)stream>>>(F, timeout_flag);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return RAFTK_OK;
}

// ---- farm system solve ----------------------------------------------------------------------------
extern "C" int raftk_system_solve_dev(int32_t n, int32_t nw, int32_t nrhs, double *Z, double *F, int32_t *info, void *stream)
{
    if (n <= 0 || nw <= 0 || nrhs <= 0 || !Z || !F) return set_err(RAFTK_EINVAL, "bad system-solve arguments");
    const size_t smem = (size_t)n * (n + nrhs) * sizeof(double2);
    if (smem > 227 * 1024) return set_err(RAFTK_EINVAL, "system too large for the shared-memory solver (n*(n+nrhs)*16 B > 227 KB)");
    static SmemOptIn opt(48 * 1024);
    CUDA_TRY(opt.ensure(k_system_solve, smem));
    k_system_solve<<<nw, 128, smem, (cudaStream_t)stream>>>(n, nrhs, reinterpret_cast<double2 *>(Z), reinterpret_cast<double2 *>(F), info);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return RAFTK_OK;
}

static int farm_launch(const raftk_designs *d, const raftk_cases *c, const raftk_outputs *solved, const raftk_farm *f, cudaStream_t st)
{
    if (!d || !c || !solved || !f) return set_err(RAFTK_EINVAL, "farm response: null argument");
    if (f->n_fowt != d->n_designs || f->n_fowt < 1) return set_err(RAFTK_EINVAL, "farm response: farm.n_fowt must equal designs.n_designs");
    if (!solved->B_drag || !solved->F_drag || !solved->F_iner || !f->Xi_sys)
        return set_err(RAFTK_EINVAL, "farm response needs B_drag, F_drag, F_iner of the per-FOWT solve and farm.Xi_sys");
    if (d->n_bem_head > 0 && !solved->F_BEM) return set_err(RAFTK_EINVAL, "farm response: the designs carry BEM excitation, F_BEM is required");
    const int n = 6 * f->n_fowt;
    const bool warp = n <= 24;                          // one warp per (frequency, case), wpc systems per CTA; at 6N = 48 it measured 13.6 ms vs 10.6 ms blocked
    const size_t sys_bytes = (size_t)n * (n + 1) * sizeof(double2);
    const int wpc = warp ? (int)std::max<size_t>(1, std::min<size_t>(FARM_WPC, (100 * 1024) / sys_bytes)) : 1;
    const size_t smem = (size_t)wpc * sys_bytes;
    if (smem > 227 * 1024) return set_err(RAFTK_EINVAL, "farm too large for the shared-memory solver (6N (6N+1) 16 B > 227 KB: N <= 19)");
    if (c->n_cases > 65535) return set_err(RAFTK_EINVAL, "farm response: more than 65535 cases per call");
    static SmemOptIn opt_w(48 * 1024), opt_b(48 * 1024);
    if (warp) CUDA_TRY(opt_w.ensure(k_farm_response<true>, smem));
    else CUDA_TRY(opt_b.ensure(k_farm_response<false>, smem));
    DesignsDev D = to_dev(d, d->max_nodes, d->max_members);
    CasesDev C = to_dev(c);
    FarmParams P;
    P.N = f->n_fowt; P.nC = c->n_cases; P.nw = d->nw;
    P.B_drag = solved->B_drag;
    P.F_drag = reinterpret_cast<const double2 *>(solved->F_drag);
    P.F_iner = reinterpret_cast<const double2 *>(solved->F_iner);
    P.F_BEM = d->n_bem_head > 0 ? reinterpret_cast<const double2 *>(solved->F_BEM) : nullptr;
    P.M_arr = f->M_arr; P.B_arr = f->B_arr; P.C_arr = f->C_arr;
    P.Xi = reinterpret_cast<double2 *>(f->Xi_sys); P.info = f->info;
    {
        ProfScope ps(st, 1);
        // 6N = 12 (the shipped two-FOWT farm): rows in registers, one lane per row, two systems per warp (k_farm_rows: 0.188 ms
        // against 0.398 ms for 65 536 systems); RAFTK_FARM_SMEM=1 keeps the shared-memory warp kernel (A/B).  At 6N = 18 / 24 the
        // register rows need 188 / 238 registers and lose (6N = 24: 2.46 ms against 1.37 ms), so those stay on the warp kernel.
        const bool rows = n == 12 && !getenv("RAFTK_FARM_SMEM");
        if (rows) k_farm_rows<12><<<dim3((d->nw + 7) / 8, c->n_cases), 128, 0, st>>>(D, C, P);
        else if (warp) k_farm_response<true><<<dim3((d->nw + wpc - 1) / wpc, c->n_cases), 32 * wpc, smem, st>>>(D, C, P);
        else k_farm_response<false><<<dim3(d->nw, c->n_cases), 256, smem, st>>>(D, C, P);
    }
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return RAFTK_OK;
}

extern "C" int raftk_farm_response_dev(const raftk_designs *d, const raftk_cases *c, const raftk_outputs *solved, const raftk_farm *f,
                                       void *stream)
{
    return farm_launch(d, c, solved, f, (cudaStream_t)stream);
}


// ---- native node-table builder for design families (pure host code, raftk_builder.h) ---------------------------------
static int set_err_i(int code, const char *fmt, int a = 0, int b = 0)
{
    snprintf(g_err, sizeof(g_err), fmt, a, b);
    return code;
}

static int family_run(const raftk_family *f, raftk_family_tables *t, int32_t *n_mem_total, int32_t *n_node_total)
{
    if (!f || f->n_designs <= 0 || f->n_members <= 0 || !f->members) return set_err(RAFTK_EINVAL, "family: empty family");
    for (int m = 0; m < f->n_members; m++) {
        const raftk_family_member &M = f->members[m];
        if (M.n_stations < 2) return set_err_i(RAFTK_EINVAL, "family: member %d: at least two stations entries must be provided", m);
        if (!M.stations || !M.rA || !M.rB || !M.d || !M.Cd_q || !M.Cd_p1 || !M.Cd_p2 || !M.Cd_End || !M.Ca_p1 || !M.Ca_p2 || !M.Ca_End)
            return set_err_i(RAFTK_EINVAL, "family: member %d: null array", m);
        if (!(M.dls_max > 0.0)) return set_err_i(RAFTK_EINVAL, "family: member %d: dls_max must be positive", m);
    }
    std::vector<rkb::MemberOut> mem(f->n_members);
    int64_t nm = 0, nn = 0;
    int max_nodes = 0, max_members = 0, mw = 0, mh = 0, mz = 0;
    if (t) t->member_offset[0] = 0, t->mem_node_start[0] = 0;
    for (int d = 0; d < f->n_designs; d++) {
        double A[36];
        for (int i = 0; i < 36; i++) A[i] = 0.0;
        int kept = 0, nodes = 0;
        for (int m = 0; m < f->n_members; m++) {
            const int rc = rkb::build_member(f->members[m], d, f->rho, f->g, f->Rp, f->r0, mem[m], A, t == nullptr);
            if (rc == -1) return set_err_i(RAFTK_EINVAL, "RAFT Members cannot start or end on the waterplane (design %d, member %d)", d, m);
            if (rc) return set_err_i(RAFTK_EINVAL, "family: the station list of member %d is not in ascending order", m);
            if (!mem[m].nodes.empty()) { kept++; nodes += (int)mem[m].nodes.size(); }
        }
        if (t) {
            for (int m = 0; m < f->n_members; m++) {
                const rkb::MemberOut &M = mem[m];
                if (M.nodes.empty()) continue;
                for (int a = 0; a < 3; a++) {
                    t->mem_frame[9 * nm + a] = M.q[a]; t->mem_frame[9 * nm + 3 + a] = M.p1[a]; t->mem_frame[9 * nm + 6 + a] = M.p2[a];
                    t->mem_rA[3 * nm + a] = M.rA[a]; t->mem_arm[3 * nm + a] = M.rA[a] - f->r0[a];
                }
                t->mem_circ[nm] = M.circ;
                for (const rkb::Node &N : M.nodes) {
                    t->node_ls[nn] = N.ls; t->node_cd_q[nn] = N.cd_q; t->node_cd_p1[nn] = N.cd_p1; t->node_cd_p2[nn] = N.cd_p2;
                    t->node_in_q[nn] = N.in_q; t->node_in_p1[nn] = N.in_p1; t->node_in_p2[nn] = N.in_p2; t->node_pa[nn] = N.pa;
                    nn++;
                }
                nm++;
                t->mem_node_start[nm] = (int32_t)nn;
            }
            t->member_offset[d + 1] = (int32_t)nm;
            for (int i = 0; i < 36; i++) t->A_morison[36 * (size_t)d + i] = A[i];
            int nW, nH, nZ;
            rkb::count_classes(mem, nW, nH, nZ);
            mw = std::max(mw, nW); mh = std::max(mh, nH); mz = std::max(mz, nZ);
        } else { nm += kept; nn += nodes; }
        max_nodes = std::max(max_nodes, nodes); max_members = std::max(max_members, kept);
        if (nn > 2000000000LL) return set_err(RAFTK_EINVAL, "family: more than 2^31 nodes");
    }
    if (n_mem_total) *n_mem_total = (int32_t)nm;
    if (n_node_total) *n_node_total = (int32_t)nn;
    if (t) {
        t->max_nodes = std::max(1, max_nodes); t->max_members = std::max(1, max_members);
        t->max_w_classes = std::max(1, mw); t->max_h_classes = std::max(1, mh); t->max_z_classes = std::max(1, mz);
    }
    return RAFTK_OK;
}

extern "C" int raftk_family_sizes(const raftk_family *f, int32_t *n_members_total, int32_t *n_nodes_total)
{
    if (!n_members_total || !n_nodes_total) return set_err(RAFTK_EINVAL, "family sizes: null output");
    return family_run(f, nullptr, n_members_total, n_nodes_total);
}

extern "C" int raftk_build_family_host(const raftk_family *f, raftk_family_tables *t)
{
    if (!t || !t->member_offset || !t->mem_node_start || !t->mem_circ || !t->mem_frame || !t->mem_rA || !t->mem_arm || !t->node_ls ||
        !t->node_cd_q || !t->node_cd_p1 || !t->node_cd_p2 || !t->node_in_q || !t->node_in_p1 || !t->node_in_p2 || !t->node_pa || !t->A_morison)
        return set_err(RAFTK_EINVAL, "family tables: null array");
    return family_run(f, t, nullptr, nullptr);
}

// ---- host-pointer front ends -------------------------------------------------------------------------

struct Arena {
    char *base = nullptr; size_t cap = 0, used = 0;
    int reserve(size_t bytes)
    {
        if (bytes <= cap) return 0;
        if (base) cudaFree(base);
        base = nullptr; cap = 0;
        if (cudaMalloc(&base, bytes) != cudaSuccess) { cudaGetLastError(); return -1; }
        cap = bytes;
        return 0;
    }
    void *take(size_t bytes) { void *p = base + used; used += align_up(bytes, 256); return p; }
};
static Arena g_arena[RAFTK_MAX_DEV];       // one per device: the *_host paths run on whichever device is current
static std::mutex g_arena_mu;

// Device scratch of the small *_host wrappers (statistics, system solve, second-order force, slender-body QTF, generalised
// DOFs): one grow-only block per device, bump-allocated per call -- no cudaMalloc / cudaFree on the call path once the
// high-water mark has been reached (SURVEY.md 8b: no hidden allocation per call).
static Arena g_scratch[RAFTK_MAX_DEV];
static std::mutex g_scratch_mu;
struct ScratchCall {
    std::unique_lock<std::mutex> lk;
    Arena &A;
    ScratchCall() : lk(g_scratch_mu), A(g_scratch[cur_dev()]) { A.used = 0; }
    bool reserve(size_t total) { return A.reserve(total + 4096) == 0; }
    template <class T> T *take(size_t bytes) { return static_cast<T *>(A.take(bytes)); }
};

// Small input arrays (grid, member/node tables, case table: ~30 arrays of a few KB) are gathered in one pinned
// staging block and sent with a single copy into a reserved region at the head of the arena; only large arrays
// (frequency tables, big sweeps) are copied one by one.  This trims ~100 us of per-copy launch overhead per call.
static const size_t SMALL_REGION = (size_t)1 << 20, SMALL_MAX = (size_t)64 << 10;
struct Stager {
    char *host = nullptr;            // pinned, SMALL_REGION bytes
    size_t used = 0;
    bool ensure()
    {
        if (host) return true;
        if (cudaHostAlloc(&host, SMALL_REGION, cudaHostAllocPortable) != cudaSuccess) { cudaGetLastError(); host = nullptr; return false; }
        return true;
    }
};
static Stager g_stage;

template <class T>
static const T *up(Arena &A, const T *h, size_t n, cudaStream_t st, cudaError_t &e)
{
    if (!h || n == 0) return nullptr;
    const size_t bytes = n * sizeof(T);
    if (bytes <= SMALL_MAX && g_stage.host && g_stage.used + align_up(bytes, 256) <= SMALL_REGION) {
        memcpy(g_stage.host + g_stage.used, h, bytes);                 // device twin: A.base + same offset
        const T *dptr = reinterpret_cast<const T *>(A.base + g_stage.used);
        g_stage.used += align_up(bytes, 256);
        return dptr;
    }
    T *dptr = static_cast<T *>(A.take(bytes));
    cudaError_t r = cudaMemcpyAsync(dptr, h, bytes, cudaMemcpyHostToDevice, st);
    if (r != cudaSuccess) e = r;
    return dptr;
}

static cudaError_t flush_small(Arena &A, cudaStream_t st)
{
    if (!g_stage.host || g_stage.used == 0) return cudaSuccess;
    return cudaMemcpyAsync(A.base, g_stage.host, g_stage.used, cudaMemcpyHostToDevice, st);
}

static size_t in_bytes(const raftk_designs *d, const raftk_cases *c)
{
    const size_t nD = d->n_designs, nw = d->nw, Nm = d->n_members_total, Ns = d->n_nodes_total, nC = c->n_cases;
    size_t b = 0;
    auto add = [&](size_t n) { b += align_up(n, 256); };
    add(nw * 8); add(nw * 8); add((nD + 1) * 4); add(Nm * 72); add(Nm * 24); add(Nm * 24); add((Nm + 1) * 4); add(Nm * 4);
    for (int t = 0; t < 8; t++) add(Ns * 8);
    if (d->node_in_p1_w) { add(Ns * nw * 16); add(Ns * nw * 16); }
    add(nD * 288); add(nD * 288); add(nD * 288);
    if (d->A_w) add(nD * 36 * nw * 8);
    if (d->B_w) add(nD * 36 * nw * 8);
    if (d->n_bem_head > 0) { add((size_t)d->n_bem_head * 8); add(nD * d->n_bem_head * 6 * nw * 16); add(nD * 24); }
    for (int t = 0; t < 4; t++) add(nC * 8);
    add(nC * 4); add(nC * 4);
    if (c->zeta) add(nC * nw * 8);
    if (c->F_2nd) add(nD * nC * 6 * nw * 8);
    if (c->Xi_init) add(nD * nC * 6 * nw * 16);
    if (d->n_qtf_w > 0) {
        add((size_t)d->n_qtf_w * 8); add((size_t)d->n_qtf_head * 8);
        add((d->qtf_shared == 1 ? 1 : (d->qtf_shared == 2 ? nD * nC : nD)) * (size_t)d->n_qtf_w * d->n_qtf_w * d->n_qtf_head * 96);
    }
    return b;
}

static int host_run(const raftk_designs *d, const raftk_cases *c, const raftk_solve_opts *o, const raftk_outputs *out,
                    const double *Xi_in, int mode, const raftk_farm *farm = nullptr)
{
    int rc = validate(d, c);
    if (rc) return rc;
    if (!out) return set_err(RAFTK_EINVAL, "null outputs");
    std::lock_guard<std::mutex> lk(g_arena_mu);
    const size_t nD = d->n_designs, nw = d->nw, nC = c->n_cases, Nm = d->n_members_total, Ns = d->n_nodes_total;
    const size_t resp = nD * nC * 6 * nw * 16;
    size_t obytes = 0;
    auto oadd = [&](const void *p, size_t n) { if (p) obytes += align_up(n, 256); };
    oadd(out->Xi, resp); oadd(out->status, nD * nC * 16); oadd(out->B_drag, nD * nC * 288); oadd(out->F_drag, resp);
    oadd(out->F_iner, resp); oadd(out->F_BEM, resp); oadd(out->zeta, nC * nw * 8); oadd(out->Xi_last, resp);
    const bool qtf_solve = (mode == 0 && d->n_qtf_w > 0 && !c->F_2nd);   // potSecOrder 2: compute the force on the device first
    if (qtf_solve) obytes += align_up(resp / 2, 256) + align_up(nD * nC * 48, 256);
    if (Xi_in) obytes += align_up(resp, 256);
    if (farm) {
        // the system response reads the per-FOWT loads on the device: those buffers exist even when the caller does not want them back
        obytes += 4 * align_up(resp, 256) + align_up(nD * nC * 288, 256) + align_up(nC * nw * 4, 256) + 3 * align_up(36 * nD * nD * 8, 256);
    }
    size_t wb = raftk_workspace_bytes(d, (int32_t)nC);
    if (mode != 0) wb = chunk_bytes((int)nD, (int)nC, d->max_nodes, (int)nw);   // single chunk required
    else {
        F2Plan f2; FPlan fp;
        if (fused2_plan(d, (int)nC, o ? o->cluster_size : 0, f2)) wb = f2.ws_bytes;
        else if (fused_plan(d, (int)(nD * nC), o ? o->cluster_size : 0, true, fp)) wb = raftk_solve_workspace_bytes(d, (int32_t)nC);
    }
    const size_t total = SMALL_REGION + in_bytes(d, c) + obytes + align_up(wb, 256) + 4096;
    Arena &A = g_arena[cur_dev()];
    if (A.reserve(total)) return set_err(RAFTK_ENOMEM, "device arena allocation failed");
    A.used = SMALL_REGION;                   // [0, SMALL_REGION) mirrors the pinned staging block
    g_stage.ensure();
    g_stage.used = 0;
    cudaStream_t st = 0;
    cudaError_t e = cudaSuccess;
    raftk_designs dd = *d;
    dd.w = up(A, d->w, nw, st, e); dd.k = up(A, d->k, nw, st, e);
    dd.member_offset = up(A, d->member_offset, nD + 1, st, e);
    dd.mem_frame = up(A, d->mem_frame, Nm * 9, st, e); dd.mem_rA = up(A, d->mem_rA, Nm * 3, st, e);
    dd.mem_arm = up(A, d->mem_arm, Nm * 3, st, e);
    dd.mem_node_start = up(A, d->mem_node_start, Nm + 1, st, e); dd.mem_circ = up(A, d->mem_circ, Nm, st, e);
    dd.node_ls = up(A, d->node_ls, Ns, st, e); dd.node_cd_q = up(A, d->node_cd_q, Ns, st, e);
    dd.node_cd_p1 = up(A, d->node_cd_p1, Ns, st, e); dd.node_cd_p2 = up(A, d->node_cd_p2, Ns, st, e);
    dd.node_in_q = up(A, d->node_in_q, Ns, st, e); dd.node_in_p1 = up(A, d->node_in_p1, Ns, st, e);
    dd.node_in_p2 = up(A, d->node_in_p2, Ns, st, e); dd.node_pa = up(A, d->node_pa, Ns, st, e);
    dd.node_in_p1_w = up(A, d->node_in_p1_w, d->node_in_p1_w ? Ns * nw * 2 : 0, st, e);
    dd.node_in_p2_w = up(A, d->node_in_p2_w, d->node_in_p2_w ? Ns * nw * 2 : 0, st, e);
    dd.M0 = up(A, d->M0, nD * 36, st, e); dd.B0 = up(A, d->B0, nD * 36, st, e); dd.C0 = up(A, d->C0, nD * 36, st, e);
    dd.A_w = up(A, d->A_w, nD * 36 * nw, st, e); dd.B_w = up(A, d->B_w, nD * 36 * nw, st, e);
    if (d->n_bem_head > 0) {
        dd.bem_headings = up(A, d->bem_headings, (size_t)d->n_bem_head, st, e);
        dd.X_BEM = up(A, d->X_BEM, nD * d->n_bem_head * 6 * nw * 2, st, e);
        dd.bem_xyh = up(A, d->bem_xyh, nD * 3, st, e);
    }
    raftk_cases cc = *c;
    cc.Hs = up(A, c->Hs, nC, st, e); cc.Tp = up(A, c->Tp, nC, st, e); cc.gamma = up(A, c->gamma, nC, st, e);
    cc.beta_deg = up(A, c->beta_deg, nC, st, e); cc.spec = up(A, c->spec, nC, st, e);
    cc.zeta = up(A, c->zeta, nC * nw, st, e);
    cc.primary = up(A, c->primary, c->primary ? nC : 0, st, e);
    cc.F_2nd = up(A, c->F_2nd, c->F_2nd ? nD * nC * 6 * nw : 0, st, e);
    cc.Xi_init = up(A, c->Xi_init, c->Xi_init ? nD * nC * 6 * nw * 2 : 0, st, e);
    if (d->n_qtf_w > 0) {
        dd.qtf_w = up(A, d->qtf_w, (size_t)d->n_qtf_w, st, e);
        dd.qtf_heads = up(A, d->qtf_heads, (size_t)d->n_qtf_head, st, e);
        dd.qtf = up(A, d->qtf, (d->qtf_shared == 1 ? 1 : (d->qtf_shared == 2 ? nD * nC : nD)) * (size_t)d->n_qtf_w * d->n_qtf_w * d->n_qtf_head * 12, st, e);
    }
    const double *Xi_in_d = up(A, Xi_in, Xi_in ? nD * nC * 6 * nw * 2 : 0, st, e);
    raftk_farm fd;
    memset(&fd, 0, sizeof(fd));
    if (farm) {                                           // array-level matrices: staged with the other small inputs
        fd = *farm;
        const size_t nn = 36 * nD * nD;
        fd.M_arr = up(A, farm->M_arr, farm->M_arr ? nn : 0, st, e);
        fd.B_arr = up(A, farm->B_arr, farm->B_arr ? nn : 0, st, e);
        fd.C_arr = up(A, farm->C_arr, farm->C_arr ? nn : 0, st, e);
    }
    {
        cudaError_t r = flush_small(A, st);
        if (r != cudaSuccess) e = r;
    }
    if (e != cudaSuccess) return set_err(RAFTK_ECUDA, "H2D copy: %s", cudaGetErrorString(e));
    raftk_outputs od;
    memset(&od, 0, sizeof(od));
    if (out->Xi) od.Xi = static_cast<double *>(A.take(resp));
    if (out->status) od.status = static_cast<int32_t *>(A.take(nD * nC * 16));
    if (out->B_drag || farm) od.B_drag = static_cast<double *>(A.take(nD * nC * 288));
    if (out->F_drag || farm) od.F_drag = static_cast<double *>(A.take(resp));
    if (out->F_iner || farm) od.F_iner = static_cast<double *>(A.take(resp));
    if (out->F_BEM || (farm && d->n_bem_head > 0)) od.F_BEM = static_cast<double *>(A.take(resp));
    if (out->zeta) od.zeta = static_cast<double *>(A.take(nC * nw * 8));
    if (out->Xi_last) od.Xi_last = static_cast<double *>(A.take(resp));
    if (qtf_solve) {
        od.F_2nd = static_cast<double *>(A.take(resp / 2));
        od.F_2nd_mean = static_cast<double *>(A.take(nD * nC * 48));
        rc = run_qtf(&dd, &cc, od.F_2nd, od.F_2nd_mean, st);
        if (rc) return rc;
        cc.F_2nd = od.F_2nd;
    }
    void *ws = A.take(wb);
    // Page-locked output buffers (raftk_host_alloc / cudaHostAlloc / cudaHostRegister): the solve kernel stores every finished
    // unit's Xi and status word straight into host memory through the unified address space -- the same epilogue that feeds
    // peer GPUs, with the host as the "peer" -- so the device-to-host transfer overlaps the units still iterating instead of
    // following the kernel as a separate copy.  RAFTK_NO_DIRECT_D2H=1 keeps the copy (A/B).
    bool direct_xi = false;
    raftk_peers hostpeer;
    if (mode == 0 && out->Xi && !getenv("RAFTK_NO_DIRECT_D2H")) {
        F2Plan f2; FPlan fp;
        const bool fused = (fused2_plan(&dd, (int)nC, o ? o->cluster_size : 0, f2) && wb >= f2.ws_bytes) ||
                           fused_plan(&dd, (int)(nD * nC), o ? o->cluster_size : 0, true, fp);
        cudaPointerAttributes pa;
        const bool pinned_xi = cudaPointerGetAttributes(&pa, out->Xi) == cudaSuccess && pa.type == cudaMemoryTypeHost && pa.devicePointer != nullptr;
        if (!pinned_xi) cudaGetLastError();
        if (fused && pinned_xi) {
            memset(&hostpeer, 0, sizeof(hostpeer));
            hostpeer.n_ranks = 2; hostpeer.rank = 0; hostpeer.epoch = 1; hostpeer.block_elems = resp / 16;
            hostpeer.gathered[0] = od.Xi;
            hostpeer.gathered[1] = static_cast<double *>(pa.devicePointer) - 0;          // block of "rank 0" inside the host array = its start
            cudaPointerAttributes ps;
            if (out->status && cudaPointerGetAttributes(&ps, out->status) == cudaSuccess && ps.type == cudaMemoryTypeHost && ps.devicePointer)
                hostpeer.status[1] = static_cast<int32_t *>(ps.devicePointer);
            else cudaGetLastError();
            direct_xi = true;
        }
    }
    if (mode == 0) rc = run(&dd, &cc, o, &od, nullptr, 0, true, ws, wb, st, direct_xi ? &hostpeer : nullptr);
    else if (mode == 2) rc = run(&dd, &cc, nullptr, &od, nullptr, 2, true, ws, wb, st);
    else {
        rc = run(&dd, &cc, nullptr, &od, nullptr, 2, true, ws, wb, st);
        if (!rc) rc = run(&dd, &cc, nullptr, &od, Xi_in_d, 1, false, ws, wb, st);
    }
    if (rc) return rc;
    if (farm) {
        fd.Xi_sys = static_cast<double *>(A.take(resp));
        fd.info = farm->info ? static_cast<int32_t *>(A.take(nC * nw * 4)) : nullptr;
        rc = farm_launch(&dd, &cc, &od, &fd, st);
        if (rc) return rc;
    }
    auto down = [&](void *h, const void *dv, size_t n) { if (h && dv) { cudaError_t r = cudaMemcpyAsync(h, dv, n, cudaMemcpyDeviceToHost, st); if (r != cudaSuccess) e = r; } };
    if (!direct_xi) down(out->Xi, od.Xi, resp);
    if (!(direct_xi && hostpeer.status[1])) down(out->status, od.status, nD * nC * 16);
    down(out->B_drag, od.B_drag, nD * nC * 288);
    down(out->F_drag, od.F_drag, resp); down(out->F_iner, od.F_iner, resp); down(out->F_BEM, od.F_BEM, resp);
    down(out->zeta, od.zeta, nC * nw * 8);
    down(out->F_2nd, od.F_2nd, resp / 2); down(out->F_2nd_mean, od.F_2nd_mean, nD * nC * 48); down(out->Xi_last, od.Xi_last, resp);
    if (farm) { down(farm->Xi_sys, fd.Xi_sys, resp); down(farm->info, fd.info, nC * nw * 4); }
    cudaError_t se = cudaStreamSynchronize(st);
    if (e != cudaSuccess || se != cudaSuccess)
        return set_err(RAFTK_ECUDA, "kernel/D2H: %s", cudaGetErrorString(se != cudaSuccess ? se : e));
    return RAFTK_OK;
}

extern "C" int raftk_hydro_excitation_host(const raftk_designs *d, const raftk_cases *c, const raftk_outputs *out)
{
    return host_run(d, c, nullptr, out, nullptr, 2);
}
extern "C" int raftk_hydro_linearization_host(const raftk_designs *d, const raftk_cases *c, const double *Xi_in, const raftk_outputs *out)
{
    if (!Xi_in) return set_err(RAFTK_EINVAL, "null Xi_in");
    return host_run(d, c, nullptr, out, Xi_in, 1);
}
extern "C" int raftk_solve_dynamics_host(const raftk_designs *d, const raftk_cases *c, const raftk_solve_opts *o, const raftk_outputs *out)
{
    if (!out || !out->Xi || !out->status || !o) return set_err(RAFTK_EINVAL, "Xi, status and opts are required");
    return host_run(d, c, o, out, nullptr, 0);
}

extern "C" int raftk_solve_dynamics_farm_host(const raftk_designs *d, const raftk_cases *c, const raftk_solve_opts *o,
                                              const raftk_outputs *out, const raftk_farm *f)
{
    if (!out || !out->Xi || !out->status || !o) return set_err(RAFTK_EINVAL, "Xi, status and opts are required");
    if (!f || !f->Xi_sys) return set_err(RAFTK_EINVAL, "farm.Xi_sys is required");
    if (d && f->n_fowt != d->n_designs) return set_err(RAFTK_EINVAL, "farm response: farm.n_fowt must equal designs.n_designs");
    return host_run(d, c, o, out, nullptr, 0, f);
}

extern "C" int raftk_second_order_force_host(const raftk_designs *d, const raftk_cases *c, const raftk_outputs *out)
{
    if (!out || !out->F_2nd) return set_err(RAFTK_EINVAL, "outputs.F_2nd is required");
    int rc = validate_qtf(d, c);
    if (rc) return rc;
    const size_t nD = d->n_designs, nw = d->nw, nC = c->n_cases, n2 = d->n_qtf_w, nh = d->n_qtf_head;
    const size_t qb = (d->qtf_shared == 1 ? 1 : (d->qtf_shared == 2 ? nD * nC : nD)) * n2 * n2 * nh * 96, fb = nD * nC * 6 * nw * 8, mb = nD * nC * 48;
    // one temporary block: grid, table axes, table, case columns, (zeta), outputs
    size_t total = 0;
    auto take = [&](size_t n) { size_t o = total; total += align_up(n, 256); return o; };
    const size_t o_w = take(nw * 8), o_qw = take(n2 * 8), o_qh = take(nh * 8), o_q = take(qb);
    const size_t o_hs = take(nC * 8), o_tp = take(nC * 8), o_ga = take(nC * 8), o_be = take(nC * 8), o_sp = take(nC * 4);
    const size_t o_ze = take(c->zeta ? nC * nw * 8 : 0), o_f = take(fb), o_m = take(mb);
    ScratchCall sc;
    if (!sc.reserve(total)) return set_err(RAFTK_ENOMEM, "second-order force: device scratch allocation failed");
    char *base = sc.take<char>(total);
    cudaError_t e = cudaSuccess;
    auto h2d = [&](size_t off, const void *h, size_t n) { if (h && n) { cudaError_t r = cudaMemcpy(base + off, h, n, cudaMemcpyHostToDevice); if (r != cudaSuccess) e = r; } };
    h2d(o_w, d->w, nw * 8); h2d(o_qw, d->qtf_w, n2 * 8); h2d(o_qh, d->qtf_heads, nh * 8); h2d(o_q, d->qtf, qb);
    h2d(o_hs, c->Hs, nC * 8); h2d(o_tp, c->Tp, nC * 8); h2d(o_ga, c->gamma, nC * 8); h2d(o_be, c->beta_deg, nC * 8);
    h2d(o_sp, c->spec, nC * 4); h2d(o_ze, c->zeta, c->zeta ? nC * nw * 8 : 0);
    raftk_designs dd = *d;
    dd.w = reinterpret_cast<double *>(base + o_w); dd.qtf_w = reinterpret_cast<double *>(base + o_qw);
    dd.qtf_heads = reinterpret_cast<double *>(base + o_qh); dd.qtf = reinterpret_cast<double *>(base + o_q);
    raftk_cases cc = *c;
    cc.Hs = reinterpret_cast<double *>(base + o_hs); cc.Tp = reinterpret_cast<double *>(base + o_tp);
    cc.gamma = reinterpret_cast<double *>(base + o_ga); cc.beta_deg = reinterpret_cast<double *>(base + o_be);
    cc.spec = reinterpret_cast<int32_t *>(base + o_sp);
    cc.zeta = c->zeta ? reinterpret_cast<double *>(base + o_ze) : nullptr;
    cc.primary = nullptr; cc.F_2nd = nullptr;
    if (e == cudaSuccess) rc = run_qtf(&dd, &cc, reinterpret_cast<double *>(base + o_f), reinterpret_cast<double *>(base + o_m), nullptr);
    if (e == cudaSuccess && !rc) {
        e = cudaMemcpy(out->F_2nd, base + o_f, fb, cudaMemcpyDeviceToHost);
        if (e == cudaSuccess && out->F_2nd_mean) e = cudaMemcpy(out->F_2nd_mean, base + o_m, mb, cudaMemcpyDeviceToHost);
    }
    if (e != cudaSuccess) return set_err(RAFTK_ECUDA, "second-order force: %s", cudaGetErrorString(e));
    return rc;
}

// ---- generalised degrees of freedom (flexible members) ---------------------------------------------------------------
struct GenLayout { size_t u, f6, Fi, Fd, XL, Bm, Bd, Z, fl, total; };
static GenLayout gen_layout(const raftk_general *g, size_t nC)
{
    const size_t n = g->n_dof, nw = g->nw, Ns = std::max(g->n_nodes, 1);
    GenLayout L; size_t t = 0;
    auto take = [&](size_t b) { size_t o = t; t += align_up(b, 256); return o; };
    L.u = take(nC * Ns * 3 * nw * 16); L.f6 = take(nC * Ns * 6 * nw * 16);
    L.Fi = take(nC * n * nw * 16); L.Fd = take(nC * n * nw * 16); L.XL = take(nC * n * nw * 16);
    L.Bm = take(nC * Ns * 9 * 8); L.Bd = take(nC * n * n * 8);
    L.Z = take(nC * nw * n * (n + 1) * 16); L.fl = take(nC * 16);
    L.total = t;
    return L;
}

extern "C" size_t raftk_general_workspace_bytes(const raftk_general *g, int32_t n_cases)
{
    if (!g || n_cases <= 0 || g->n_dof <= 0 || g->nw <= 0) return 0;
    return gen_layout(g, (size_t)n_cases).total;
}

extern "C" int raftk_general_solve_dynamics_dev(const raftk_general *g, const raftk_cases *c, const raftk_solve_opts *o, double *Xi,
                                                int32_t *status, void *workspace, size_t workspace_bytes, void *stream)
{
    if (!g || !c || !o || !Xi || !status) return set_err(RAFTK_EINVAL, "general solve: null argument");
    if (g->n_dof <= 0 || g->n_dof > 256 || g->nw <= 0 || g->n_nodes < 0 || c->n_cases <= 0 || c->n_cases > 65535)
        return set_err(RAFTK_EINVAL, "general solve: 0 < n_dof <= 256, nw > 0, 0 < n_cases <= 65535");
    if (c->primary || c->F_2nd || c->Xi_init) return set_err(RAFTK_EINVAL, "general solve: wave trains / F_2nd / Xi_init are not supported");
    const size_t nC = c->n_cases;
    const GenLayout L = gen_layout(g, nC);
    if (!workspace || workspace_bytes < L.total) return set_err(RAFTK_ENOMEM, "general solve: workspace too small");
    GenDev D;
    D.n = g->n_dof; D.nw = g->nw; D.Ns = g->n_nodes; D.depth = g->depth; D.dw = g->dw; D.rho = g->rho;
    D.w = g->w; D.k = g->k; D.node_r = g->node_r; D.node_frame = g->node_frame; D.node_circ = g->node_circ;
    D.node_Imat = g->node_Imat; D.node_Imat_w = reinterpret_cast<const double2 *>(g->node_Imat_w);
    D.node_a_i = g->node_a_i; D.node_cd = g->node_cd; D.Tn = g->Tn; D.rr = g->rr; D.M = g->M; D.B = g->B; D.C = g->C;
    char *b = static_cast<char *>(workspace);
    GenWork W;
    W.u = reinterpret_cast<double2 *>(b + L.u); W.f6 = reinterpret_cast<double2 *>(b + L.f6);
    W.F_iner = reinterpret_cast<double2 *>(b + L.Fi); W.F_drag = reinterpret_cast<double2 *>(b + L.Fd);
    W.XiLast = reinterpret_cast<double2 *>(b + L.XL); W.Bmat = reinterpret_cast<double *>(b + L.Bm);
    W.B_drag = reinterpret_cast<double *>(b + L.Bd); W.Z = reinterpret_cast<double2 *>(b + L.Z); W.flags = reinterpret_cast<int *>(b + L.fl);
    CasesDev C = to_dev(c);
    cudaStream_t st = (cudaStream_t)stream;
    double2 *X = reinterpret_cast<double2 *>(Xi);
    const unsigned fb = (unsigned)((g->nw + 127) / 128);
    // blocked LU (panel + row block in shared memory); RAFTK_GEN_UNBLOCKED=1 keeps the first, column-at-a-time kernel for A/B runs
    const size_t lu_smem = ((size_t)g->n_dof * GB + (size_t)GB * (g->n_dof + 1)) * sizeof(double2);
    const bool blocked = !getenv("RAFTK_GEN_UNBLOCKED") && lu_smem <= 110 * 1024;
    if (blocked) {
        static SmemOptIn opt(48 * 1024);
        CUDA_TRY(opt.ensure(k_gen_solve_blocked, lu_smem));
    }
    prof_begin_call();
    k_gen_init<<<(unsigned)nC, 256, 0, st>>>(D, W, o->xi_start);
    if (g->n_nodes > 0) k_gen_wave<<<dim3(fb, g->n_nodes, (unsigned)nC), 128, 0, st>>>(D, C, W);
    k_gen_project<<<dim3(fb, g->n_dof, (unsigned)nC), 128, 0, st>>>(D, W, W.F_iner, 0);
    g_launches += 3;
    for (int pass = 0; pass < o->n_iter + 1; pass++) {
        if (g->n_nodes > 0) k_gen_node_pass<<<dim3(g->n_nodes, (unsigned)nC), 128, 0, st>>>(D, W);
        k_gen_bdrag<<<dim3(g->n_dof, (unsigned)nC), 128, 0, st>>>(D, W);
        k_gen_project<<<dim3(fb, g->n_dof, (unsigned)nC), 128, 0, st>>>(D, W, W.F_drag, 1);
        if (blocked) {
            ProfScope ps(st, 2);
            k_gen_solve_blocked<<<dim3(g->nw, (unsigned)nC), GT, lu_smem, st>>>(D, W, X, o->tol);
        } else {
            ProfScope ps(st, 2);
            k_gen_solve<<<dim3(g->nw, (unsigned)nC), 256, 0, st>>>(D, W, X, o->tol);
        }
        k_gen_relax<<<(unsigned)nC, 256, 0, st>>>(D, W, X);
        g_launches += 5;
    }
    k_gen_status<<<(unsigned)((nC + 127) / 128), 128, 0, st>>>((int)nC, W.flags, status);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return RAFTK_OK;
}

extern "C" int raftk_general_solve_dynamics_host(const raftk_general *g, const raftk_cases *c, const raftk_solve_opts *o, double *Xi,
                                                 int32_t *status)
{
    if (!g || !c || !o || !Xi || !status) return set_err(RAFTK_EINVAL, "general solve: null argument");
    if (g->n_dof <= 0 || g->nw <= 0 || c->n_cases <= 0) return set_err(RAFTK_EINVAL, "general solve: empty problem");
    const size_t n = g->n_dof, nw = g->nw, Ns = g->n_nodes, nC = c->n_cases;
    size_t total = 0;
    auto take = [&](size_t b) { size_t o_ = total; total += align_up(std::max<size_t>(b, 8), 256); return o_; };
    raftk_general gg = *g; raftk_cases cc = *c;
    struct Item { size_t off; const void *h; size_t nb; const void **slot; };
    std::vector<Item> items;
    auto add = [&](const void *h, size_t nb, const void **slot) { if (h) items.push_back({take(nb), h, nb, slot}); };
    add(g->w, nw * 8, (const void **)&gg.w); add(g->k, nw * 8, (const void **)&gg.k);
    add(g->node_r, Ns * 24, (const void **)&gg.node_r); add(g->node_frame, Ns * 72, (const void **)&gg.node_frame);
    add(g->node_circ, Ns * 4, (const void **)&gg.node_circ); add(g->node_Imat, Ns * 72, (const void **)&gg.node_Imat);
    add(g->node_Imat_w, Ns * 9 * nw * 16, (const void **)&gg.node_Imat_w); add(g->node_a_i, Ns * 8, (const void **)&gg.node_a_i);
    add(g->node_cd, Ns * 32, (const void **)&gg.node_cd); add(g->Tn, Ns * 6 * n * 8, (const void **)&gg.Tn); add(g->rr, Ns * 24, (const void **)&gg.rr);
    add(g->M, n * n * 8, (const void **)&gg.M); add(g->B, n * n * 8, (const void **)&gg.B); add(g->C, n * n * 8, (const void **)&gg.C);
    add(c->Hs, nC * 8, (const void **)&cc.Hs); add(c->Tp, nC * 8, (const void **)&cc.Tp); add(c->gamma, nC * 8, (const void **)&cc.gamma);
    add(c->beta_deg, nC * 8, (const void **)&cc.beta_deg); add(c->spec, nC * 4, (const void **)&cc.spec); add(c->zeta, nC * nw * 8, (const void **)&cc.zeta);
    const size_t o_xi = take(nC * n * nw * 16), o_st = take(nC * 16);
    const size_t wb = raftk_general_workspace_bytes(g, (int32_t)nC), o_ws = take(wb);
    ScratchCall sc;
    if (!sc.reserve(total)) return set_err(RAFTK_ENOMEM, "general solve: device scratch allocation failed");
    char *base = sc.take<char>(total);
    for (auto &it : items) { CUDA_TRY(cudaMemcpy(base + it.off, it.h, it.nb, cudaMemcpyHostToDevice)); *it.slot = base + it.off; }
    int rc = raftk_general_solve_dynamics_dev(&gg, &cc, o, reinterpret_cast<double *>(base + o_xi), reinterpret_cast<int32_t *>(base + o_st),
                                              base + o_ws, wb, nullptr);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpy(Xi, base + o_xi, nC * n * nw * 16, cudaMemcpyDeviceToHost));
    CUDA_TRY(cudaMemcpy(status, base + o_st, nC * 16, cudaMemcpyDeviceToHost));
    return RAFTK_OK;
}

// ---- slender-body QTF ----------------------------------------------------------------------------------
static int validate_slender(const raftk_slender *s, int32_t n_cases)
{
    if (!s || n_cases <= 0 || s->nw <= 0 || s->n_members <= 0 || s->n_nodes < 0 || s->n_seg < 0)
        return set_err(RAFTK_EINVAL, "bad slender-body QTF arguments (n_cases, nw, n_members must be > 0)");
    if (n_cases > 65535) return set_err(RAFTK_EINVAL, "slender-body QTF: more than 65535 cases per call");
    return 0;
}

extern "C" size_t raftk_qtf_slender_workspace_bytes(const raftk_slender *s, int32_t n_cases)
{
    if (!s || n_cases <= 0) return 0;
    return align_up((size_t)n_cases * std::max(s->n_nodes, 1) * s->nw * SL_NODE_C * sizeof(cx), 256)
           + align_up((size_t)n_cases * s->n_members * s->nw * SL_MEM_C * sizeof(cx), 256)
           + align_up((size_t)(s->n_members + s->n_seg) * s->nw * SL_HANK * sizeof(cx), 256);
}

extern "C" int raftk_qtf_slender_dev(const raftk_slender *s, int32_t n_cases, const double *beta_rad, const double *Xi_rao, double *qtf,
                                     void *workspace, size_t workspace_bytes, void *stream)
{
    int rc = validate_slender(s, n_cases);
    if (rc) return rc;
    if (!beta_rad || !Xi_rao || !qtf) return set_err(RAFTK_EINVAL, "slender-body QTF: null beta / Xi_rao / qtf");
    if (!workspace || workspace_bytes < raftk_qtf_slender_workspace_bytes(s, n_cases)) return set_err(RAFTK_ENOMEM, "slender-body QTF: workspace too small");
    SlenderDev D;
    D.n_nodes = s->n_nodes; D.n_members = s->n_members; D.n_seg = s->n_seg; D.nw = s->nw;
    D.depth = s->depth; D.rho = s->rho; D.g = s->g;
    D.mem_q = s->mem_q; D.mem_p1 = s->mem_p1; D.mem_p2 = s->mem_p2; D.mem_mcf = s->mem_mcf; D.mem_wl = s->mem_wl;
    D.mem_r_int = s->mem_r_int; D.mem_a_wl = s->mem_a_wl; D.mem_rwl = s->mem_rwl; D.mem_R_wl = s->mem_R_wl;
    D.mem_node_start = s->mem_node_start; D.node_r = s->node_r; D.node_v_side = s->node_v_side;
    D.node_Ca_p1 = s->node_Ca_p1; D.node_Ca_p2 = s->node_Ca_p2; D.node_Ca_End = s->node_Ca_End; D.node_v_end = s->node_v_end; D.node_a_i = s->node_a_i;
    D.seg_mem = s->seg_mem; D.seg_z1 = s->seg_z1; D.seg_z2 = s->seg_z2; D.seg_R = s->seg_R; D.seg_rmid = s->seg_rmid;
    D.M_struc = s->M_struc; D.w = s->w; D.k = s->k;
    cudaStream_t st = (cudaStream_t)stream;
    cx *Tn = static_cast<cx *>(workspace);
    cx *Tm = reinterpret_cast<cx *>(static_cast<char *>(workspace) + align_up((size_t)n_cases * std::max(s->n_nodes, 1) * s->nw * SL_NODE_C * sizeof(cx), 256));
    cx *Th = reinterpret_cast<cx *>(reinterpret_cast<char *>(Tm) + align_up((size_t)n_cases * s->n_members * s->nw * SL_MEM_C * sizeof(cx), 256));
    const cx *X = reinterpret_cast<const cx *>(Xi_rao);
    cx *Q = reinterpret_cast<cx *>(qtf);
    k_slender_tables<<<dim3(s->n_nodes + 2 * s->n_members + s->n_seg, n_cases), SL_THREADS, 0, st>>>(D, beta_rad, X, Tn, Tm, Th);
    const unsigned npairs = (unsigned)((size_t)s->nw * (s->nw + 1) / 2);
    k_slender_pairs<<<dim3(npairs, n_cases), SL_THREADS, 0, st>>>(D, beta_rad, X, Tn, Tm, Th, Q);
    k_slender_fill<<<dim3(s->nw, n_cases), 64, 0, st>>>(s->nw, Q);
    g_launches += 3;
    CUDA_TRY(cudaGetLastError());
    return RAFTK_OK;
}

extern "C" int raftk_qtf_slender_host(const raftk_slender *s, int32_t n_cases, const double *beta_rad, const double *Xi_rao, double *qtf)
{
    int rc = validate_slender(s, n_cases);
    if (rc) return rc;
    if (!beta_rad || !Xi_rao || !qtf) return set_err(RAFTK_EINVAL, "slender-body QTF: null beta / Xi_rao / qtf");
    const size_t Nm = s->n_members, Ns = s->n_nodes, Ng = s->n_seg, nw = s->nw, nC = n_cases;
    size_t total = 0;
    auto take = [&](size_t n) { size_t o = total; total += align_up(std::max<size_t>(n, 8), 256); return o; };
    struct Item { size_t off; const void *h; size_t n; const void **slot; };
    raftk_slender dd = *s;
    std::vector<Item> items;
    auto add = [&](const void *h, size_t n, const void **slot) { items.push_back({take(n), h, n, slot}); };
    add(s->w, nw * 8, (const void **)&dd.w); add(s->k, nw * 8, (const void **)&dd.k);
    add(s->mem_q, Nm * 24, (const void **)&dd.mem_q); add(s->mem_p1, Nm * 24, (const void **)&dd.mem_p1); add(s->mem_p2, Nm * 24, (const void **)&dd.mem_p2);
    add(s->mem_mcf, Nm * 4, (const void **)&dd.mem_mcf); add(s->mem_wl, Nm * 4, (const void **)&dd.mem_wl);
    add(s->mem_r_int, Nm * 24, (const void **)&dd.mem_r_int); add(s->mem_a_wl, Nm * 8, (const void **)&dd.mem_a_wl);
    add(s->mem_rwl, Nm * 24, (const void **)&dd.mem_rwl); add(s->mem_R_wl, Nm * 8, (const void **)&dd.mem_R_wl);
    add(s->mem_node_start, (Nm + 1) * 4, (const void **)&dd.mem_node_start);
    add(s->node_r, Ns * 24, (const void **)&dd.node_r); add(s->node_v_side, Ns * 8, (const void **)&dd.node_v_side);
    add(s->node_Ca_p1, Ns * 8, (const void **)&dd.node_Ca_p1); add(s->node_Ca_p2, Ns * 8, (const void **)&dd.node_Ca_p2);
    add(s->node_Ca_End, Ns * 8, (const void **)&dd.node_Ca_End); add(s->node_v_end, Ns * 8, (const void **)&dd.node_v_end);
    add(s->node_a_i, Ns * 8, (const void **)&dd.node_a_i);
    add(s->seg_mem, Ng * 4, (const void **)&dd.seg_mem); add(s->seg_z1, Ng * 8, (const void **)&dd.seg_z1); add(s->seg_z2, Ng * 8, (const void **)&dd.seg_z2);
    add(s->seg_R, Ng * 8, (const void **)&dd.seg_R); add(s->seg_rmid, Ng * 24, (const void **)&dd.seg_rmid);
    add(s->M_struc, 288, (const void **)&dd.M_struc);
    const size_t o_beta = take(nC * 8), o_xi = take(nC * 6 * nw * 16), o_q = take(nC * nw * nw * 6 * 16);
    const size_t wb = raftk_qtf_slender_workspace_bytes(s, n_cases), o_ws = take(wb);
    ScratchCall sc;
    if (!sc.reserve(total)) return set_err(RAFTK_ENOMEM, "slender-body QTF: device scratch allocation failed");
    char *base = sc.take<char>(total);
    cudaError_t e = cudaSuccess;
    for (auto &it : items) {
        if (it.h && it.n) { cudaError_t r = cudaMemcpy(base + it.off, it.h, it.n, cudaMemcpyHostToDevice); if (r != cudaSuccess) e = r; }
        *it.slot = base + it.off;
    }
    if (e == cudaSuccess) e = cudaMemcpy(base + o_beta, beta_rad, nC * 8, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) e = cudaMemcpy(base + o_xi, Xi_rao, nC * 6 * nw * 16, cudaMemcpyHostToDevice);
    if (e == cudaSuccess) {
        rc = raftk_qtf_slender_dev(&dd, n_cases, reinterpret_cast<double *>(base + o_beta), reinterpret_cast<double *>(base + o_xi),
                                   reinterpret_cast<double *>(base + o_q), base + o_ws, wb, nullptr);
        if (!rc) e = cudaMemcpy(qtf, base + o_q, nC * nw * nw * 6 * 16, cudaMemcpyDeviceToHost);
    }
    if (e != cudaSuccess) return set_err(RAFTK_ECUDA, "slender-body QTF: %s", cudaGetErrorString(e));
    return rc;
}

extern "C" int raftk_system_solve_host(int32_t n, int32_t nw, int32_t nrhs, double *Z, double *F, int32_t *info)
{
    if (n <= 0 || nw <= 0 || nrhs <= 0 || !Z || !F) return set_err(RAFTK_EINVAL, "bad system-solve arguments");
    const size_t zb = (size_t)nw * n * n * 16, fb = (size_t)nw * n * nrhs * 16, ib = (size_t)nw * 4;
    ScratchCall sc;
    if (!sc.reserve(align_up(zb, 256) + align_up(fb, 256) + align_up(ib, 256))) return set_err(RAFTK_ENOMEM, "system solve: device scratch allocation failed");
    double *dZ = sc.take<double>(zb), *dF = sc.take<double>(fb);
    int32_t *dI = sc.take<int32_t>(ib);
    CUDA_TRY(cudaMemcpy(dZ, Z, zb, cudaMemcpyHostToDevice)); CUDA_TRY(cudaMemcpy(dF, F, fb, cudaMemcpyHostToDevice));
    int rc = raftk_system_solve_dev(n, nw, nrhs, dZ, dF, dI, nullptr);
    if (!rc) {
        CUDA_TRY(cudaMemcpy(F, dF, fb, cudaMemcpyDeviceToHost));
        if (info) CUDA_TRY(cudaMemcpy(info, dI, ib, cudaMemcpyDeviceToHost));
    }
    return rc;
}

extern "C" int raftk_response_stats_dev(int32_t n_units, int32_t nw, double dw, int32_t rot_deg, const double *Xi,
                                        double *sd, double *psd, void *stream)
{
    if (n_units <= 0 || nw <= 0 || !Xi || !sd || !(dw > 0.0)) return set_err(RAFTK_EINVAL, "bad response-stats arguments");
    k_response_stats<<<(unsigned)n_units * 6u, 128, 0, (cudaStream_t)stream>>>(nw, dw, rot_deg, reinterpret_cast<const double2 *>(Xi), sd, psd);
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return RAFTK_OK;
}

extern "C" int raftk_response_stats_host(int32_t n_units, int32_t nw, double dw, int32_t rot_deg, const double *Xi,
                                         double *sd, double *psd)
{
    if (n_units <= 0 || nw <= 0 || !Xi || !sd || !(dw > 0.0)) return set_err(RAFTK_EINVAL, "bad response-stats arguments");
    const size_t xb = (size_t)n_units * 6 * nw * 16, sb = (size_t)n_units * 6 * 8, pb = (size_t)n_units * 6 * nw * 8;
    ScratchCall sc;
    if (!sc.reserve(align_up(xb, 256) + align_up(sb, 256) + align_up(pb, 256))) return set_err(RAFTK_ENOMEM, "response stats: device scratch allocation failed");
    double *dX = sc.take<double>(xb), *dS = sc.take<double>(sb), *dP = psd ? sc.take<double>(pb) : nullptr;
    CUDA_TRY(cudaMemcpy(dX, Xi, xb, cudaMemcpyHostToDevice));
    int rc = raftk_response_stats_dev(n_units, nw, dw, rot_deg, dX, dS, dP, nullptr);
    if (!rc) {
        CUDA_TRY(cudaMemcpy(sd, dS, sb, cudaMemcpyDeviceToHost));
        if (psd) CUDA_TRY(cudaMemcpy(psd, dP, pb, cudaMemcpyDeviceToHost));
    }
    return rc;
}

extern "C" int raftk_channel_stats_dev(int32_t n_designs, int32_t n_cases, int32_t n_ch, int32_t nw, double dw, const double *coef,
                                       const double *Xi, double *sd, double *psd, double *amp, void *stream)
{
    if (n_designs <= 0 || n_cases <= 0 || n_ch <= 0 || nw <= 0 || !coef || !Xi || !sd || !(dw > 0.0))
        return set_err(RAFTK_EINVAL, "bad channel-stats arguments");
    const size_t rows = (size_t)n_designs * n_cases * n_ch;
    if (rows > 2147483647u) return set_err(RAFTK_EINVAL, "channel-stats: too many (design, case, channel) rows");
    k_channel_stats<<<(unsigned)rows, 128, 0, (cudaStream_t)stream>>>(n_cases, n_ch, nw, dw, reinterpret_cast<const double2 *>(coef),
                                                                    reinterpret_cast<const double2 *>(Xi), sd, psd, reinterpret_cast<double2 *>(amp));
    g_launches++;
    CUDA_TRY(cudaGetLastError());
    return RAFTK_OK;
}

extern "C" int raftk_channel_stats_host(int32_t n_designs, int32_t n_cases, int32_t n_ch, int32_t nw, double dw, const double *coef,
                                        const double *Xi, double *sd, double *psd, double *amp)
{
    if (n_designs <= 0 || n_cases <= 0 || n_ch <= 0 || nw <= 0 || !coef || !Xi || !sd || !(dw > 0.0))
        return set_err(RAFTK_EINVAL, "bad channel-stats arguments");
    const size_t rows = (size_t)n_designs * n_cases * n_ch;
    const size_t cb = (size_t)n_designs * n_ch * 6 * nw * 16, xb = (size_t)n_designs * n_cases * 6 * nw * 16;
    const size_t sb = rows * 8, pb = rows * nw * 8, ab = rows * nw * 16;
    ScratchCall sc;
    if (!sc.reserve(align_up(cb, 256) + align_up(xb, 256) + align_up(sb, 256) + align_up(pb, 256) + align_up(ab, 256)))
        return set_err(RAFTK_ENOMEM, "channel stats: device scratch allocation failed");
    double *dC = sc.take<double>(cb), *dX = sc.take<double>(xb), *dS = sc.take<double>(sb);
    double *dP = psd ? sc.take<double>(pb) : nullptr, *dA = amp ? sc.take<double>(ab) : nullptr;
    CUDA_TRY(cudaMemcpy(dC, coef, cb, cudaMemcpyHostToDevice)); CUDA_TRY(cudaMemcpy(dX, Xi, xb, cudaMemcpyHostToDevice));
    int rc = raftk_channel_stats_dev(n_designs, n_cases, n_ch, nw, dw, dC, dX, dS, dP, dA, nullptr);
    if (!rc) {
        CUDA_TRY(cudaMemcpy(sd, dS, sb, cudaMemcpyDeviceToHost));
        if (psd) CUDA_TRY(cudaMemcpy(psd, dP, pb, cudaMemcpyDeviceToHost));
        if (amp) CUDA_TRY(cudaMemcpy(amp, dA, ab, cudaMemcpyDeviceToHost));
    }
    return rc;
}

extern "C" void *raftk_host_alloc(size_t bytes)
{
    void *p = nullptr;
    if (cudaHostAlloc(&p, bytes, cudaHostAllocDefault) != cudaSuccess) { cudaGetLastError(); return nullptr; }
    return p;
}
extern "C" void raftk_host_free(void *p) { if (p) cudaFreeHost(p); }

extern "C" double raftk_fp64_peak_gflops(int iters)
{
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    const int blocks = sms * 8, threads = 256;
    double *out = nullptr;
    if (cudaMalloc(&out, (size_t)blocks * threads * 8) != cudaSuccess) return -1.0;
    cudaEvent_t a, b;
    cudaEventCreate(&a); cudaEventCreate(&b);
    k_fp64_peak<<<blocks, threads>>>(out, 1000);
    cudaDeviceSynchronize();
    cudaEventRecord(a);
    k_fp64_peak<<<blocks, threads>>>(out, iters);
    cudaEventRecord(b);
    cudaEventSynchronize(b);
    g_launches += 2;
    float ms = 0;
    cudaEventElapsedTime(&ms, a, b);
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(out);
    const double flops = 2.0 * 8.0 * (double)iters * blocks * threads;
    return flops / (ms * 1e-3) * 1e-9;
}
