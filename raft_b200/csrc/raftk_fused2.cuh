// raftk_fused2.cuh -- k_fused_plan + k_rao_fused2: second generation of the fused on-chip solver (included by raftk.cu only).
//
// Same algorithm and recurrences as k_rao_fused (raftk_fused.cuh); what changed is the mapping, driven by the measured FP64
// pipe (profiles/r02_fp64_micro.txt: DFMA latency 8.2 cycles, one warp instruction per 2 cycles per scheduler; with the two
// resident warps per scheduler that 254 registers allow, the pipe saturates only at >= 2 independent chains per thread):
//   * TWO frequency bins per thread.  The node walks of both bins are interleaved instruction by instruction (two
//     independent E/A recurrences -> ILP 2); the per-node RMS accumulators, the linearised coefficients and the step-class
//     indices are shared by both bins, so the warp reductions, the coefficient loads and the address arithmetic per bin halve.
//     A CTA of 128 threads owns 256 bins: cfg2 runs as ONE wave of 4-CTA clusters instead of 1.73 waves of 8-CTA clusters.
//   * the per-design tables (member frames and lever arms, node columns, system matrices, step classes with every node's
//     factor-table offsets) are built ONCE per design by k_fused_plan into a 16-byte aligned blob and staged into shared
//     memory by ONE TMA bulk copy (cp.async.bulk + mbarrier) instead of being rebuilt with scalar loads by every CTA.
//   * per-bin shared memory is down to the step-factor tables and the iterate (256 B per bin for VolturnUS-S): member base
//     phases / depth pairs and the linear excitation live in the L2-resident workspace and are prefetched one member ahead;
//     the walking-state checkpoint between node chunks stays in registers.
#pragma once

#define F2_T 128                 // threads per CTA (4 warps, 2 CTAs per SM at 254 registers)
#define F2_TRW 8                 // values per round of the transposed warp reduction

struct PlanLayout {
    int o_mem, o_node, nstr, o_mat, o_wkey, o_hkey, o_zkey, o_rec, o_int, total;   // offsets / sizes in doubles
    int i_imem, i_nodem, i_cnt, i_chunk, n_int;                                    // offsets in ints from o_int
};

__host__ __device__ inline PlanLayout plan_layout(int NmP, int NsP, int maxW, int maxH, int maxZ)
{
    PlanLayout L;
    int p = 0;
    L.o_mem = p; p += NmP * MEM_STRIDE;        // per member: frame (9), a x d (9), [18..20] heading projections (per case), z0, x0, y0
    L.nstr = (NsP + 1) & ~1;
    L.o_node = p; p += 8 * L.nstr;             // node columns: ls, cd_q, cd_p1, cd_p2, in_q, in_p1, in_p2, pa
    L.o_mat = p; p += 108;                     // M0, B0, C0
    L.o_wkey = p; p += 2 * maxW;
    L.o_hkey = p; p += maxH;
    L.o_zkey = p; p += maxZ;
    p = (p + 1) & ~1;
    L.o_rec = p; p += 2 * (NsP + 12);          // node records {ls, factor-table offsets}; +12: the node walk prefetches up to 10 entries ahead
    L.o_int = p;
    int q = 0;
    L.i_imem = q; q += NmP * IMEM_STRIDE;
    L.i_nodem = q; q += NsP + 12;
    L.i_cnt = q; q += 4;                       // nW, nH, overflow, nZ
    L.i_chunk = q; q += 2 * ((NsP + CHUNK_NODES - 1) / CHUNK_NODES);   // per chunk of the RMS walk: direction mask, reduction-round mask
    q = (q + 3) & ~3;
    L.n_int = q;
    L.total = p + q / 2;                       // even number of doubles -> a multiple of 16 bytes
    return L;
}

// ------------------------------------------------------------------------------------------------
// k_fused_plan: one CTA per design.  Stages the design's tables and builds the step classes (distinct node spacings
// (q_x,q_y)*step and q_z*step, distinct first-node depths) exactly as k_rao_fused does per CTA, once, into the blob.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_fused_plan(DesignsDev D, double *plan, size_t stride, int maxW, int maxH, int maxZ, int nwl)
{
    extern __shared__ __align__(16) double smem_raw[];
    const int d = blockIdx.x, tid = threadIdx.x, T = blockDim.x;
    const int m0 = D.member_offset[d], Nm = D.member_offset[d + 1] - m0;
    const int nbase = D.mem_node_start[m0];
    const int Ns = D.mem_node_start[m0 + Nm] - nbase;
    const int NsP = D.max_nodes, NmP = D.max_members;
    const PlanLayout L = plan_layout(NmP, NsP, maxW, maxH, maxZ);
    double *blob = plan + (size_t)d * stride;
    double *mem = blob + L.o_mem, *node = blob + L.o_node, *mat = blob + L.o_mat;
    double *wkey = blob + L.o_wkey, *hkey = blob + L.o_hkey, *zkey = blob + L.o_zkey;
    int *ib = reinterpret_cast<int *>(blob + L.o_int);
    int *imem = ib + L.i_imem, *node_m = ib + L.i_nodem, *cnt_g = ib + L.i_cnt;
    double2 *rec = reinterpret_cast<double2 *>(blob + L.o_rec);
    double *scr = smem_raw;                                   // 3 * NsP key components
    double *z0s = scr + 3 * (size_t)NsP;                      // NmP first-node depths
    int *iscr = reinterpret_cast<int *>(z0s + NmP);           // 2 * NsP representatives
    int *mstart = iscr + 2 * NsP;                             // 2 * NmP member node ranges
    __shared__ int cnt[4];
    if (tid < 4) cnt[tid] = 0;
    for (int t = tid; t < L.total; t += T) blob[t] = 0.0;
    __syncthreads();
    for (int m = tid; m < Nm; m += T) {
        const double *fr = D.mem_frame + 9 * (m0 + m);
        const double *arm = D.mem_arm + 3 * (m0 + m);
        const double *rA = D.mem_rA + 3 * (m0 + m);
        double *o = mem + m * MEM_STRIDE;
        for (int t = 0; t < 9; t++) o[t] = fr[t];
        for (int v = 0; v < 3; v++) {
            const double d0_ = fr[3 * v], d1_ = fr[3 * v + 1], d2_ = fr[3 * v + 2];
            o[9 + 3 * v + 0] = arm[1] * d2_ - arm[2] * d1_;
            o[9 + 3 * v + 1] = arm[2] * d0_ - arm[0] * d2_;
            o[9 + 3 * v + 2] = arm[0] * d1_ - arm[1] * d0_;
        }
        const int js = D.mem_node_start[m0 + m] - nbase, je = D.mem_node_start[m0 + m + 1] - nbase;
        imem[IMEM_STRIDE * m + 0] = js;
        imem[IMEM_STRIDE * m + 1] = je;
        imem[IMEM_STRIDE * m + 2] = D.mem_circ[m0 + m];
        mstart[2 * m] = js; mstart[2 * m + 1] = je;
        const double ls0 = D.node_ls[nbase + js];
        const double z0 = rA[2] + ls0 * fr[2];
        o[21] = z0; o[22] = rA[0] + ls0 * fr[0]; o[23] = rA[1] + ls0 * fr[1];
        z0s[m] = z0;
    }
    for (int j = tid; j < Ns; j += T) {
        node[0 * L.nstr + j] = D.node_ls[nbase + j];
        node[1 * L.nstr + j] = D.node_cd_q[nbase + j];
        node[2 * L.nstr + j] = D.node_cd_p1[nbase + j];
        node[3 * L.nstr + j] = D.node_cd_p2[nbase + j];
        node[4 * L.nstr + j] = D.node_in_q[nbase + j];
        node[5 * L.nstr + j] = D.node_in_p1[nbase + j];
        node[6 * L.nstr + j] = D.node_in_p2[nbase + j];
        node[7 * L.nstr + j] = D.node_pa[nbase + j];
    }
    for (int t = tid; t < 36; t += T) {
        mat[t] = D.M0[(size_t)d * 36 + t];
        mat[36 + t] = D.B0[(size_t)d * 36 + t];
        mat[72 + t] = D.C0[(size_t)d * 36 + t];
    }
    __syncthreads();
    // A: keys per node
    for (int j = tid; j < Ns; j += T) {
        int m = 0;
        while (j >= mstart[2 * m + 1]) m++;
        node_m[j] = m;
        const double *fr = D.mem_frame + 9 * (m0 + m);
        double kx = 0, ky = 0, kz = 0;
        if (j > mstart[2 * m]) {
            const double step = D.node_ls[nbase + j] - D.node_ls[nbase + j - 1];
            kx = fr[0] * step; ky = fr[1] * step; kz = fr[2] * step;
        }
        scr[j] = kx; scr[NsP + j] = ky; scr[2 * NsP + j] = kz;
    }
    __syncthreads();
    // B: representative (first node with the same key)
    for (int j = tid; j < Ns; j += T) {
        const double kx = scr[j], ky = scr[NsP + j], kz = scr[2 * NsP + j];
        int rw = -1, rh = -1;
        if (fabs(kx) > 1e-14 || fabs(ky) > 1e-14) {
            const double tol = 1e-11 * (fabs(kx) + fabs(ky));
            rw = j;
            for (int x = 0; x < j; x++)
                if (fabs(scr[x] - kx) <= tol && fabs(scr[NsP + x] - ky) <= tol) { rw = x; break; }
        }
        if (fabs(kz) > 1e-14) {
            const double tol = 1e-11 * fabs(kz);
            rh = j;
            for (int x = 0; x < j; x++)
                if (fabs(scr[2 * NsP + x] - kz) <= tol) { rh = x; break; }
        }
        iscr[j] = rw; iscr[NsP + j] = rh;
    }
    __syncthreads();
    // C: class id = rank of the representative among representatives; offsets into the factor tables (class * nwl).  A
    // node's record holds its position ls and its phase / depth offsets (as the low / high word of the second double), so
    // the walks fetch everything a node step needs from the plan with one 16-byte load
    for (int j = tid; j < Ns; j += T) {
        const int rw = iscr[j], rh = iscr[NsP + j];
        int wi = -1, hi = -1;
        if (rw >= 0) { wi = 0; for (int x = 0; x < rw; x++) wi += (iscr[x] == x); }
        if (rh >= 0) { hi = 0; for (int x = 0; x < rh; x++) hi += (iscr[NsP + x] == x); }
        if (wi >= maxW) { wi = 0; cnt[2] = 1; }
        if (hi >= maxH) { hi = 0; cnt[2] = 1; }
        if (rw == j && wi >= 0) { wkey[2 * wi] = scr[j]; wkey[2 * wi + 1] = scr[NsP + j]; atomicMax(&cnt[0], wi + 1); }
        if (rh == j && hi >= 0) { hkey[hi] = scr[2 * NsP + j]; atomicMax(&cnt[1], hi + 1); }
        // identity row when the phase / depth does not change
        rec[j] = make_double2(D.node_ls[nbase + j], __hiloint2double((hi >= 0 ? hi : maxH) * nwl, (wi >= 0 ? wi : maxW) * nwl));
    }
    for (int j = Ns + tid; j < NsP + 12; j += T) {
        rec[j] = make_double2(0.0, __hiloint2double(maxH * nwl, maxW * nwl));
        node_m[j] = Nm > 0 ? Nm - 1 : 0;
    }
    // z classes of the members' first nodes
    for (int m = tid; m < Nm; m += T) {
        const double z0 = z0s[m];
        int rep = m;
        for (int x = 0; x < m; x++) if (fabs(z0s[x] - z0) <= 1e-12 * fmax(1.0, fabs(z0))) { rep = x; break; }
        int zi = 0;
        for (int x = 0; x < rep; x++) {
            const double zx = z0s[x];
            bool first = true;
            for (int y = 0; y < x; y++) if (fabs(z0s[y] - zx) <= 1e-12 * fmax(1.0, fabs(zx))) { first = false; break; }
            zi += first;
        }
        if (zi >= maxZ) { zi = 0; cnt[2] = 1; }
        if (rep == m) { zkey[zi] = z0; atomicMax(&cnt[3], zi + 1); }
        imem[IMEM_STRIDE * m + 4] = zi;
    }
    // drag-direction masks per chunk of CHUNK_NODES nodes.  The reference's strips carry axial drag only where a member ends
    // or steps (Cd_End, raft_member.py:2098-2117) and transverse drag only where the strip has a length, so most nodes need
    // one or two of the three relative-velocity projections: a direction whose coefficient is exactly zero contributes an
    // exact zero to B_drag / F_drag and is skipped.  Node jj of a chunk: bit 3jj = axial, bit 3jj+1 = transverse.
    // Accumulator slots of a chunk: [0,10) = transverse-1 (or axial when the node has no transverse drag), [10,20) =
    // transverse-2, [20,30) = axial of a node that has both; the round mask says which 8-value reduction rounds hold any.
    {
        int *chunk_g = ib + L.i_chunk;
        const int nchunk = (NsP + CHUNK_NODES - 1) / CHUNK_NODES;
        for (int ch = tid; ch < nchunk; ch += T) {
            unsigned cm = 0, slots = 0;
            for (int jj = 0; jj < CHUNK_NODES; jj++) {
                const int j = ch * CHUNK_NODES + jj;
                if (j >= Ns) break;
                const bool q = D.node_cd_q[nbase + j] != 0.0;
                const bool p = D.node_cd_p1[nbase + j] != 0.0 || D.node_cd_p2[nbase + j] != 0.0;
                cm |= ((q ? 1u : 0u) | (p ? 2u : 0u)) << (3 * jj);
                if (q || p) slots |= 1u << jj;
                if (p) slots |= 1u << (10 + jj);
                if (q && p) slots |= 1u << (20 + jj);
            }
            unsigned rm = 0;
            for (int rd = 0; rd < 4; rd++) if ((slots >> (rd * F2_TRW)) & 0xffu) rm |= 1u << rd;
            chunk_g[2 * ch] = (int)cm;
            chunk_g[2 * ch + 1] = (int)rm;
        }
    }
    __syncthreads();
    if (tid < 4) cnt_g[tid] = cnt[tid];
}

// ------------------------------------------------------------------------------------------------
// TMA / mbarrier helpers (sm_90+ PTX; the bulk copy is the non-tensor form: one contiguous, 16-byte aligned block)
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ unsigned smem_u32(const void *p) { return (unsigned)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(unsigned long long *bar, unsigned count)
{
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_expect_tx(unsigned long long *bar, unsigned bytes)
{
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_g2s(void *dst, const void *src, unsigned bytes, unsigned long long *bar)
{
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(smem_u32(dst)), "l"(src), "r"(bytes), "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(unsigned long long *bar, unsigned parity)
{
    asm volatile("{\n .reg .pred p;\n WAIT_%=:\n mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n @p bra DONE_%=;\n bra WAIT_%=;\n DONE_%=:\n}"
                 ::"r"(smem_u32(bar)), "r"(parity) : "memory");
}

// one copy of the slow-path-carrying libm routines: the prologue calls them from several loops, and the pass loop's code
// (node walks, reductions, 6x6 LU: ~120 KB of SASS) should stay resident in the instruction cache
__device__ __noinline__ void sincos_once(double x, double *s, double *c) { sincos(x, s, c); }
__device__ __noinline__ double exp_once(double x) { return exp(x); }
// two-argument forms for the thread's two bins: the two evaluations are independent, so their polynomial chains can overlap
__device__ __noinline__ double4 sincos2_once(double x0, double x1)
{
    double s0, c0, s1, c1;
    sincos(x0, &s0, &c0);
    sincos(x1, &s1, &c1);
    return make_double4(c0, s0, c1, s1);
}
__device__ __noinline__ double4 exp2pm_once(double a0, double a1) { return make_double4(exp(a0), exp(-a0), exp(a1), exp(-a1)); }
__device__ __noinline__ double4 depth2_once(double k0, double k1, double h, double z)
{
    double s0, c0, p0, s1, c1, p1;
    depth_funcs(k0, h, z, s0, c0, p0);
    depth_funcs(k1, h, z, s1, c1, p1);
    return make_double4(0.5 * (c0 + s0), 0.5 * (c0 - s0), 0.5 * (c1 + s1), 0.5 * (c1 - s1));
}
__device__ __noinline__ double jonswap_once(double w, double Hs, double Tp, double Gamma) { return jonswap(w, Hs, Tp, Gamma); }
// sea_state_zeta (raftk_tables.cuh) with the spectrum evaluated out of line
__device__ __forceinline__ double zeta_f2(const CasesDev &Cs, int c, int i, int nw, double w, double dw)
{
    if (Cs.zeta_in) return Cs.zeta_in[(size_t)c * nw + i];
    const int spec = Cs.spec[c];
    double S = 0.0;
    if (spec == RAFTK_SPEC_JONSWAP) S = jonswap_once(w, Cs.Hs[c], Cs.Tp[c], Cs.gamma[c]);
    else if (spec == RAFTK_SPEC_UNIT) S = 1.0;
    else if (spec == RAFTK_SPEC_CONSTANT) S = Cs.Hs[c];
    return sqrt(2.0 * S * dw);
}
__device__ __noinline__ void depth_once(double k, double h, double z, double *S_, double *C_)
{
    double s, c, pd;
    depth_funcs(k, h, z, s, c, pd);
    *S_ = s; *C_ = c;
}

__host__ __device__ inline size_t fused2_smem_bytes(int Nm, int NsP, int nchunk, int nwl, int maxW, int maxH, int maxZ)
{
    const PlanLayout L = plan_layout(Nm, NsP, maxW, maxH, maxZ);
    const int nwarps = F2_T / 32;
    size_t dbl = (size_t)L.total + NCOEF * (size_t)NsP + (size_t)Nm * 8 + 36 + (size_t)nchunk * nwarps * 32 + 2 * ((size_t)nchunk * 32 + 2)
                 + (size_t)nchunk * 32 + (size_t)nwarps * F2_TRW * 33 + 2;
    dbl += 2 * ((size_t)(maxW + 1) + (maxH + 1)) * nwl + 12 * (size_t)nwl;
    return dbl * sizeof(double) + 64;
}

// |d| < tol (|x| + tol)  <=>  d.d < (tol (|x| + tol))^2 : the convergence test of raft_model.py:1103 with one square root
__device__ __forceinline__ bool conv_ok(double dr, double di, double xr, double xi, double tol)
{
    const double a = fma(dr, dr, di * di), b = fma(xr, xr, xi * xi);
    const double rhs = tol * (sqrt(b) + tol);
    return a < rhs * rhs;
}

// FULL = false: the instantiation for calls without BEM added mass / damping tables (A_w, B_w), F_drag or Xi_last outputs
// and without the primary-case hand-over (lin_g); those paths are compiled out of its pass loop, which keeps the loop's
// code (instruction-cache footprint) smaller.  The host selects it from the inputs (run_fused2 in raftk.cu).
template <bool FULL>
__global__ void __launch_bounds__(F2_T, 2)
k_rao_fused2(DesignsDev D, CasesDev Cs, FusedParams P)
{
    extern __shared__ __align__(16) double smem_raw[];
    __shared__ __align__(8) unsigned long long mbar;
    constexpr int T = F2_T, nwarps = F2_T / 32;
    __shared__ int s_flw[nwarps];
    cg::cluster_group cluster = cg::this_cluster();
    const int CS = P.CS;
    const int rank = (CS > 1) ? (int)cluster.block_rank() : 0;
    const int unit = blockIdx.x / CS;
    const int d = unit / Cs.nC, c = unit % Cs.nC;
    const int nw = D.nw, tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int prim = (FULL && P.phase >= 0 && Cs.primary) ? Cs.primary[c] : c;
    const bool secondary = prim != c;
    if ((P.phase == 0 && secondary) || (P.phase == 1 && !secondary)) return;

    const int NsP = D.max_nodes, NmP = D.max_members;
    const int nchunk = (NsP + CHUNK_NODES - 1) / CHUNK_NODES;
    const int nwl = P.nwl;
    const int f_begin = rank * nwl;
    const int nloc = max(0, min(nwl, nw - f_begin));
    const PlanLayout L = plan_layout(NmP, NsP, P.maxW, P.maxH, P.maxZ);

    double *blob = smem_raw;
    double *s_mem = blob + L.o_mem, *s_node = blob + L.o_node, *s_mat = blob + L.o_mat;
    const double *s_wkey = blob + L.o_wkey, *s_hkey = blob + L.o_hkey, *s_zkey = blob + L.o_zkey;
    const int *ib = reinterpret_cast<const int *>(blob + L.o_int);
    const int *s_imem = ib + L.i_imem, *s_nodem = ib + L.i_nodem, *s_cnt = ib + L.i_cnt;
    const double2 *s_rec = reinterpret_cast<const double2 *>(blob + L.o_rec);  // per node: ls, factor-table offsets (F2_OW / F2_OH)
#define F2_OW(R) __double2loint((R).y)
#define F2_OH(R) __double2hiint((R).y)
    const int *s_chunk = ib + L.i_chunk;
    double *p = blob + L.total;
    double *s_coef = p; p += NCOEF * (size_t)NsP;
    double *s_msum = p; p += (size_t)NmP * 8;
    double *s_bmat = p; p += 36;
    double *s_wpart = p; p += (size_t)nchunk * nwarps * 32;
    double *s_sums = p; p += 2 * ((size_t)nchunk * 32 + 2);
    double *s_tot = p; p += (size_t)nchunk * 32;
    double *s_trans = p; p += (size_t)nwarps * F2_TRW * 33;
    p += ((p - smem_raw) & 1);
    double2 *s_wtab = reinterpret_cast<double2 *>(p); p += 2 * (size_t)(P.maxW + 1) * nwl;
    double2 *s_htab = reinterpret_cast<double2 *>(p); p += 2 * (size_t)(P.maxH + 1) * nwl;
    double *s_xi = p;
    const int sums_stride = nchunk * 32 + 2;
    const int nstr = L.nstr;
    const double *n_ls = s_node, *n_cdq = s_node + nstr, *n_cd1 = s_node + 2 * nstr, *n_cd2 = s_node + 3 * nstr;
    const double *n_inq = s_node + 4 * nstr, *n_in1 = s_node + 5 * nstr, *n_in2 = s_node + 6 * nstr, *n_pa = s_node + 7 * nstr;

    // ---- stage the design's plan blob with one TMA bulk copy -----------------------------------------------------------
    if (tid == 0) mbar_init(&mbar, 1);
    __syncthreads();
    if (tid == 0) {
        const unsigned bytes = (unsigned)L.total * 8u;
        mbar_expect_tx(&mbar, bytes);
        tma_bulk_g2s(blob, P.plan + (size_t)d * P.plan_stride, bytes, &mbar);
    }
    const double beta = Cs.beta_deg[c] * (CUDART_PI / 180.0);
    double sb, cb;
    sincos(beta, &sb, &cb);
    mbar_wait(&mbar, 0);
    const int m0 = D.member_offset[d], Nm = D.member_offset[d + 1] - m0;
    const int nbase = D.mem_node_start[m0];
    const int Ns = D.mem_node_start[m0 + Nm] - nbase;
    for (int m = tid; m < Nm; m += T) {                       // heading projections of the member frame: per case
        double *o = s_mem + m * MEM_STRIDE;
        for (int v = 0; v < 3; v++) o[18 + v] = o[3 * v] * cb + o[3 * v + 1] * sb;
    }
    __syncthreads();
    const int nW = s_cnt[0], nH = s_cnt[1], nZ = s_cnt[3];
    const bool plan_overflow = s_cnt[2] != 0;
    for (int t = tid; t < nchunk * nwarps * 32; t += T) s_wpart[t] = 0.0;      // reduction rounds without an active direction are never written

    const size_t ogl = ((size_t)d * Cs.nC + c) * 6 * nw;
    double2 *Eg = P.Eg + ((size_t)d * Cs.nC + c) * (size_t)NmP * nw;      // member base phases   [NmP][nw]
    double2 *Ag = P.Ag + ((size_t)d * Cs.nC + c) * (size_t)P.maxZ * nw;   // first-node depth pairs [maxZ][nw]

    // the two bins of this thread: local indices t0 = tid, t1 = tid + T.  A bin beyond the slice is walked with a zero wave
    // amplitude and a zero iterate (contributes exact zeros to the sums) and is skipped in the solve phase.
    const bool ok0 = tid < nloc, ok1 = tid + T < nloc;
    const int t0 = ok0 ? tid : 0, t1 = ok1 ? tid + T : t0;
    const int ibase = nloc > 0 ? f_begin : 0;                 // a CTA beyond the grid still reads in-range table entries
    const int i0 = ibase + t0, i1 = ibase + t1;
    const double w0 = ok0 ? D.w[i0] : 0.0, w1 = ok1 ? D.w[i1] : 0.0;
    const double2 *wtA = s_wtab + t0, *wtB = s_wtab + t1, *htA = s_htab + t0, *htB = s_htab + t1;
    const double2 zero2 = make_double2(0.0, 0.0);

    // ---- prologue (a): sea state, step-class factors, member base phases / depth pairs; the transcendental functions of the
    //      thread's two bins are evaluated pairwise ---------------------------------------------------------------------------
    if (!plan_overflow && ok0) {
        const double kA = D.k[i0], kB = D.k[i1];
        const double zetaA = zeta_f2(Cs, c, i0, nw, D.w[i0], D.dw);
        const double zetaB = ok1 ? zeta_f2(Cs, c, i1, nw, D.w[i1], D.dw) : 0.0;
        if (P.zeta_out && d == 0) { P.zeta_out[(size_t)c * nw + i0] = zetaA; if (ok1) P.zeta_out[(size_t)c * nw + i1] = zetaB; }
        const double zwA = zetaA * w0, zwB = zetaB * w1;
#pragma unroll 1
        for (int x = 0; x < nW; x++) {
            const double g = s_wkey[2 * x] * cb + s_wkey[2 * x + 1] * sb;
            const double4 v = sincos2_once(-(kA * g), -(kB * g));
            s_wtab[x * nwl + t0] = make_double2(v.x, v.y);
            if (ok1) s_wtab[x * nwl + t1] = make_double2(v.z, v.w);
        }
#pragma unroll 1
        for (int x = 0; x < nH; x++) {
            const double4 v = exp2pm_once(kA * s_hkey[x], kB * s_hkey[x]);
            s_htab[x * nwl + t0] = make_double2(v.x, v.y);
            if (ok1) s_htab[x * nwl + t1] = make_double2(v.z, v.w);
        }
        s_wtab[P.maxW * nwl + t0] = make_double2(1.0, 0.0);
        s_htab[P.maxH * nwl + t0] = make_double2(1.0, 1.0);
        if (ok1) { s_wtab[P.maxW * nwl + t1] = make_double2(1.0, 0.0); s_htab[P.maxH * nwl + t1] = make_double2(1.0, 1.0); }
#pragma unroll 1
        for (int x = 0; x < nZ; x++) {
            const double4 v = depth2_once(kA, kB, D.depth, s_zkey[x]);
            Ag[(size_t)x * nw + i0] = make_double2(v.x, v.y);
            if (ok1) Ag[(size_t)x * nw + i1] = make_double2(v.z, v.w);
        }
#pragma unroll 1
        for (int m = 0; m < Nm; m++) {
            const double *o = s_mem + m * MEM_STRIDE;
            const double g = cb * o[22] + sb * o[23];
            const double4 v = sincos2_once(-(kA * g), -(kB * g));
            Eg[(size_t)m * nw + i0] = make_double2(zwA * v.x, zwA * v.y);
            if (ok1) Eg[(size_t)m * nw + i1] = make_double2(zwB * v.z, zwB * v.w);
        }
#pragma unroll
        for (int a = 0; a < 6; a++) {
            if (P.Xi_init) {
                const double2 x0 = P.Xi_init[ogl + (size_t)a * nw + i0];
                s_xi[(2 * a) * nwl + t0] = x0.x; s_xi[(2 * a + 1) * nwl + t0] = x0.y;
                if (ok1) { const double2 x1 = P.Xi_init[ogl + (size_t)a * nw + i1]; s_xi[(2 * a) * nwl + t1] = x1.x; s_xi[(2 * a + 1) * nwl + t1] = x1.y; }
            } else {
                s_xi[(2 * a) * nwl + t0] = P.xi_start; s_xi[(2 * a + 1) * nwl + t0] = 0.0;
                if (ok1) { s_xi[(2 * a) * nwl + t1] = P.xi_start; s_xi[(2 * a + 1) * nwl + t1] = 0.0; }
            }
        }
    }

    // ---- prologue (b): strip inertial + dynamic-pressure excitation F0, node walk of both bins interleaved -----------------
    if (!plan_overflow) {
        const double kA = D.k[i0], kB = D.k[i1];
        const bool deepA = kA * D.depth > 89.4, deepB = kB * D.depth > 89.4;
        const double thA = tanh(kA * D.depth), thB = tanh(kB * D.depth);
        double FrA[6], FiA[6], FrB[6], FiB[6];
#pragma unroll
        for (int a = 0; a < 6; a++) { FrA[a] = 0.0; FiA[a] = 0.0; FrB[a] = 0.0; FiB[a] = 0.0; }
        const bool mcf = D.node_in_p1_w != nullptr;
        for (int m = 0; m < Nm; m++) {
            const double *o = s_mem + m * MEM_STRIDE;
            const int j0 = s_imem[IMEM_STRIDE * m], j1 = s_imem[IMEM_STRIDE * m + 1], zc = s_imem[IMEM_STRIDE * m + 4];
            const double ls0 = n_ls[j0];
            const double2 eA = ok0 ? Eg[(size_t)m * nw + i0] : zero2, eB = ok1 ? Eg[(size_t)m * nw + i1] : zero2;
            const double2 aA = Ag[(size_t)zc * nw + i0], aB = Ag[(size_t)zc * nw + i1];
            double erA = eA.x, eiA = eA.y, apA = aA.x, amA = aA.y, erB = eB.x, eiB = eB.y, apB = aB.x, amB = aB.y;
            const double hq = o[18], h1 = o[19], h2 = o[20];
            double AqrA = 0, AqiA = 0, A1rA = 0, A1iA = 0, A2rA = 0, A2iA = 0, L1rA = 0, L1iA = 0, L2rA = 0, L2iA = 0;
            double AqrB = 0, AqiB = 0, A1rB = 0, A1iB = 0, A2rB = 0, A2iB = 0, L1rB = 0, L1iB = 0, L2rB = 0, L2iB = 0;
            for (int j = j0; j < j1; j++) {
                const double2 rj = s_rec[j];
                const double2 WA = wtA[F2_OW(rj)], HA = htA[F2_OH(rj)], WB = wtB[F2_OW(rj)], HB = htB[F2_OH(rj)];
                { const double tr = fma(erA, WA.x, -eiA * WA.y); eiA = fma(erA, WA.y, eiA * WA.x); erA = tr; }
                { const double tr = fma(erB, WB.x, -eiB * WB.y); eiB = fma(erB, WB.y, eiB * WB.x); erB = tr; }
                apA *= HA.x; amA *= HA.y; apB *= HB.x; amB *= HB.y;
                const double inq = n_inq[j], pa = n_pa[j], in1 = n_in1[j], in2 = n_in2[j], ls = n_ls[j];
                if (!mcf && inq == 0.0 && in1 == 0.0 && in2 == 0.0 && pa == 0.0) continue;       // potMod strip: drag only
#define F2_F0_NODE(ER, EI, AP, AM, WW, KK, II, TH, DEEP, AQR, AQI, A1R, A1I, A2R, A2I, L1R, L1I, L2R, L2I)                     \
    {                                                                                                                             \
        double i1r = in1, i1i = 0.0, i2r = in2, i2i = 0.0;                                                                        \
        if (mcf) {                                                                                                                \
            const size_t jg = (size_t)(nbase + j);                                                                                \
            const double2 v1 = D.node_in_p1_w[jg * nw + II], v2 = D.node_in_p2_w[jg * nw + II];                                   \
            i1r = v1.x; i1i = v1.y; i2r = v2.x; i2i = v2.y;                                                                        \
        }                                                                                                                         \
        const double Cc = AP + AM, Sc = AP - AM;                                                                                  \
        double cr, ci;                                                                                                            \
        proj(ER, EI, Cc, Sc, hq, o[2], cr, ci);                                                                                   \
        double fqr = -WW * inq * ci, fqi = WW * inq * cr;                                                                         \
        proj(ER, EI, Cc, Sc, h1, o[5], cr, ci);                                                                                   \
        const double f1r = -WW * (i1r * ci + i1i * cr), f1i = WW * (i1r * cr - i1i * ci);                                         \
        proj(ER, EI, Cc, Sc, h2, o[8], cr, ci);                                                                                   \
        const double f2r = -WW * (i2r * ci + i2i * cr), f2i = WW * (i2r * cr - i2i * ci);                                         \
        if (pa != 0.0 && WW != 0.0) {                                                                                             \
            double Pd = Cc * TH;                                                                                                  \
            if (DEEP) Pd = Cc + exp_once(-KK * (o[21] + (ls - ls0) * o[2] + 2.0 * D.depth));                                      \
            const double sc = pa * Pd / WW;                                                                                       \
            fqr = fma(sc, ER, fqr); fqi = fma(sc, EI, fqi);                                                                       \
        }                                                                                                                         \
        AQR += fqr; AQI += fqi; A1R += f1r; A1I += f1i; A2R += f2r; A2I += f2i;                                                   \
        L1R += ls * f1r; L1I += ls * f1i; L2R += ls * f2r; L2I += ls * f2i;                                                       \
    }
                F2_F0_NODE(erA, eiA, apA, amA, w0, kA, i0, thA, deepA, AqrA, AqiA, A1rA, A1iA, A2rA, A2iA, L1rA, L1iA, L2rA, L2iA)
                F2_F0_NODE(erB, eiB, apB, amB, w1, kB, i1, thB, deepB, AqrB, AqiB, A1rB, A1iB, A2rB, A2iB, L1rB, L1iB, L2rB, L2iB)
#undef F2_F0_NODE
            }
#pragma unroll
            for (int a = 0; a < 3; a++) {
                FrA[a] += o[a] * AqrA + o[3 + a] * A1rA + o[6 + a] * A2rA;
                FiA[a] += o[a] * AqiA + o[3 + a] * A1iA + o[6 + a] * A2iA;
                FrA[3 + a] += o[9 + a] * AqrA + o[12 + a] * A1rA + o[15 + a] * A2rA + o[6 + a] * L1rA - o[3 + a] * L2rA;
                FiA[3 + a] += o[9 + a] * AqiA + o[12 + a] * A1iA + o[15 + a] * A2iA + o[6 + a] * L1iA - o[3 + a] * L2iA;
                FrB[a] += o[a] * AqrB + o[3 + a] * A1rB + o[6 + a] * A2rB;
                FiB[a] += o[a] * AqiB + o[3 + a] * A1iB + o[6 + a] * A2iB;
                FrB[3 + a] += o[9 + a] * AqrB + o[12 + a] * A1rB + o[15 + a] * A2rB + o[6 + a] * L1rB - o[3 + a] * L2rB;
                FiB[3 + a] += o[9 + a] * AqiB + o[12 + a] * A1iB + o[15 + a] * A2iB + o[6 + a] * L1iB - o[3 + a] * L2iB;
            }
        }
        // per bin: optional outputs, BEM excitation, second-order forces; the sum is parked in the workspace
#pragma unroll 1
        for (int bsel = 0; bsel < 2; bsel++) {
            if (!(bsel == 0 ? ok0 : ok1)) continue;
            const int i = bsel == 0 ? i0 : i1;
            double Fr[6], Fi[6];
#pragma unroll
            for (int a = 0; a < 6; a++) { Fr[a] = bsel == 0 ? FrA[a] : FrB[a]; Fi[a] = bsel == 0 ? FiA[a] : FiB[a]; }
            if (P.Finer_out)
                for (int a = 0; a < 6; a++) P.Finer_out[ogl + (size_t)a * nw + i] = make_double2(Fr[a], Fi[a]);
            if (D.n_bem_head > 0) {
                const double k = D.k[i], w = D.w[i];
                const double zeta = zeta_f2(Cs, c, i, nw, w, D.dw);
                double Br[6], Bi[6];
                bem_excitation(D, d, i, k, beta, sb, cb, zeta, Br, Bi);
#pragma unroll
                for (int a = 0; a < 6; a++) {
                    if (P.Fbem_out) P.Fbem_out[ogl + (size_t)a * nw + i] = make_double2(Br[a], Bi[a]);
                    Fr[a] += Br[a]; Fi[a] += Bi[a];
                }
            } else if (P.Fbem_out) {
                for (int a = 0; a < 6; a++) P.Fbem_out[ogl + (size_t)a * nw + i] = make_double2(0.0, 0.0);
            }
            if (Cs.F_2nd) {
#pragma unroll
                for (int a = 0; a < 6; a++) Fr[a] += Cs.F_2nd[ogl + (size_t)a * nw + i];
            }
#pragma unroll
            for (int a = 0; a < 6; a++) P.F0g[ogl + (size_t)a * nw + i] = make_double2(Fr[a], Fi[a]);
        }
    }
    if (plan_overflow) {
        for (int t = tid; t < nloc; t += T)
            for (int a = 0; a < 6; a++) P.Xi_out[ogl + (size_t)a * nw + f_begin + t] = make_double2(0.0, 0.0);
    }
    __syncthreads();

    const double *Aw = FULL && D.A_w ? D.A_w + (size_t)d * 36 * nw : nullptr;
    const double *Bw = FULL && D.B_w ? D.B_w + (size_t)d * 36 * nw : nullptr;
    int passes = 0, converged = 0, flags = plan_overflow ? RAFTK_FLAG_PLAN : 0, par = 0;
    const int max_pass = plan_overflow ? 0 : (secondary ? 1 : P.n_iter + 1);
    const size_t lin_stride = (size_t)NCOEF * NsP + 36;
    if (secondary && !plan_overflow) {
        const double *src = P.lin_g + ((size_t)d * Cs.nC + prim) * lin_stride;
#pragma unroll 1
        for (int t = tid; t < NCOEF * NsP; t += T) s_coef[t] = src[t];
#pragma unroll 1
        for (int t = tid; t < 36; t += T) s_bmat[t] = src[NCOEF * NsP + t];
        __syncthreads();
    }


    for (int it = 0; it < max_pass; it++) {
        if (!secondary) {
        // ================= pass part 1: sum_w |v_rel . d|^2 per node and direction, both bins interleaved ===========
        double erA = 0, eiA = 0, apA = 0, amA = 0, erB = 0, eiB = 0, apB = 0, amB = 0;      // walking state, kept across chunks
        // member-level projections of the body velocity, -i w (d . Xi_t + (a x d) . Xi_r), per bin: computed when a member is
        // entered at its first node and kept across a chunk boundary that falls inside the member
        double mqrA = 0, mqiA = 0, m1rA = 0, m1iA = 0, m2rA = 0, m2iA = 0, u1rA = 0, u1iA = 0, u2rA = 0, u2iA = 0;
        double mqrB = 0, mqiB = 0, m1rB = 0, m1iB = 0, m2rB = 0, m2iB = 0, u1rB = 0, u1iB = 0, u2rB = 0, u2iB = 0;
        for (int ch = 0; ch < nchunk; ch++) {
            double acc[32];
#pragma unroll
            for (int t = 0; t < 32; t++) acc[t] = 0.0;
            const int jc0 = ch * CHUNK_NODES;
            const unsigned cmask = (unsigned)s_chunk[2 * ch], rmask = (unsigned)s_chunk[2 * ch + 1];
            if (jc0 < Ns) {
                int jj = 0;
                while (jj < CHUNK_NODES && jc0 + jj < Ns) {
                    const int jfirst = jc0 + jj;
                    const int mcur = s_nodem[jfirst];
                    const int mstart = s_imem[IMEM_STRIDE * mcur], jlast = s_imem[IMEM_STRIDE * mcur + 1] - jc0;
                    const double *o = s_mem + mcur * MEM_STRIDE;
#define F2_MEMBER_PROJ(TT, WW, OKK, MQR, MQI, M1R, M1I, M2R, M2I, U1R, U1I, U2R, U2I)                                          \
    {                                                                                                                             \
        double xr[6], xi[6];                                                                                                      \
        _Pragma("unroll") for (int a = 0; a < 6; a++) {                                                                           \
            xr[a] = OKK ? s_xi[(2 * a) * nwl + TT] : 0.0; xi[a] = OKK ? s_xi[(2 * a + 1) * nwl + TT] : 0.0;                      \
        }                                                                                                                         \
        double sr, si;                                                                                                            \
        sr = o[0] * xr[0] + o[1] * xr[1] + o[2] * xr[2] + o[9] * xr[3] + o[10] * xr[4] + o[11] * xr[5];                           \
        si = o[0] * xi[0] + o[1] * xi[1] + o[2] * xi[2] + o[9] * xi[3] + o[10] * xi[4] + o[11] * xi[5];                           \
        MQR = WW * si; MQI = -WW * sr;                                                                                            \
        sr = o[3] * xr[0] + o[4] * xr[1] + o[5] * xr[2] + o[12] * xr[3] + o[13] * xr[4] + o[14] * xr[5];                          \
        si = o[3] * xi[0] + o[4] * xi[1] + o[5] * xi[2] + o[12] * xi[3] + o[13] * xi[4] + o[14] * xi[5];                          \
        M1R = WW * si; M1I = -WW * sr;                                                                                            \
        sr = o[6] * xr[0] + o[7] * xr[1] + o[8] * xr[2] + o[15] * xr[3] + o[16] * xr[4] + o[17] * xr[5];                          \
        si = o[6] * xi[0] + o[7] * xi[1] + o[8] * xi[2] + o[15] * xi[3] + o[16] * xi[4] + o[17] * xi[5];                          \
        M2R = WW * si; M2I = -WW * sr;                                                                                            \
        sr = o[3] * xr[3] + o[4] * xr[4] + o[5] * xr[5];                                                                          \
        si = o[3] * xi[3] + o[4] * xi[4] + o[5] * xi[5];                                                                          \
        U1R = WW * si; U1I = -WW * sr;                                                                                            \
        sr = o[6] * xr[3] + o[7] * xr[4] + o[8] * xr[5];                                                                          \
        si = o[6] * xi[3] + o[7] * xi[4] + o[8] * xi[5];                                                                          \
        U2R = WW * si; U2I = -WW * sr;                                                                                            \
    }
                    if (jfirst == mstart) {
                        F2_MEMBER_PROJ(t0, w0, ok0, mqrA, mqiA, m1rA, m1iA, m2rA, m2iA, u1rA, u1iA, u2rA, u2iA)
                        F2_MEMBER_PROJ(t1, w1, ok1, mqrB, mqiB, m1rB, m1iB, m2rB, m2iB, u1rB, u1iB, u2rB, u2iB)
                    }
#undef F2_MEMBER_PROJ
                    const double hq = o[18], h1 = o[19], h2 = o[20], dzq = o[2], dz1 = o[5], dz2 = o[8];
                    if (jfirst == mstart) {
                        const int zc = s_imem[IMEM_STRIDE * mcur + 4];
                        const double2 eA = ok0 ? Eg[(size_t)mcur * nw + i0] : zero2, aA = Ag[(size_t)zc * nw + i0];
                        const double2 eB = ok1 ? Eg[(size_t)mcur * nw + i1] : zero2, aB = Ag[(size_t)zc * nw + i1];
                        erA = eA.x; eiA = eA.y; apA = aA.x; amA = aA.y;
                        erB = eB.x; eiB = eB.y; apB = aB.x; amB = aB.y;
                    }
                    // node body, both bins: the step factors of node JJ were loaded one node earlier (C set), those of node
                    // JJ+1 are requested first (N set); sets alternate with the parity of JJ
#define F2_STEP_BIN(ER, EI, AP, AM, CW, CH, CC, SC)                                                                              \
    { const double tr = fma(ER, CW.x, -EI * CW.y); EI = fma(ER, CW.y, EI * CW.x); ER = tr; }                                      \
    AP *= CH.x; AM *= CH.y;                                                                                                       \
    const double CC = AP + AM, SC = AP - AM;
#define F2_SQ(ER, EI, CC, SC, HH, DZ, MR, MI, OUT)                                                                                \
    { double ar_, ai_; proj_add(ER, EI, CC, SC, HH, DZ, MR, MI, ar_, ai_); OUT = fma(ar_, ar_, ai_ * ai_); }
#define F2_P1_NODE(JJ, CWA, CHA, CWB, CHB, CL, NWA, NHA, NWB, NHB, NL)                                                           \
    {                                                                                                                             \
        const int jn = jc0 + JJ + 1;                                                                                              \
        const double2 rn = s_rec[jn];                                                                                             \
        NWA = wtA[F2_OW(rn)]; NHA = htA[F2_OH(rn)]; NWB = wtB[F2_OW(rn)]; NHB = htB[F2_OH(rn)]; NL = rn.x;                        \
        const double ls = CL;                                                                                                     \
        F2_STEP_BIN(erA, eiA, apA, amA, CWA, CHA, CcA, ScA)                                                                       \
        F2_STEP_BIN(erB, eiB, apB, amB, CWB, CHB, CcB, ScB)                                                                       \
        const bool has_p = (cmask & (2u << (3 * JJ))) != 0u;                                                                      \
        if (has_p) {                                                                                                              \
            double pA, rA_, pB, rB_;                                                                                              \
            F2_SQ(erA, eiA, CcA, ScA, h1, dz1, fma(ls, u2rA, m1rA), fma(ls, u2iA, m1iA), pA)                                      \
            F2_SQ(erB, eiB, CcB, ScB, h1, dz1, fma(ls, u2rB, m1rB), fma(ls, u2iB, m1iB), pB)                                      \
            F2_SQ(erA, eiA, CcA, ScA, h2, dz2, fma(-ls, u1rA, m2rA), fma(-ls, u1iA, m2iA), rA_)                                   \
            F2_SQ(erB, eiB, CcB, ScB, h2, dz2, fma(-ls, u1rB, m2rB), fma(-ls, u1iB, m2iB), rB_)                                   \
            acc[JJ] += pA + pB; acc[10 + JJ] += rA_ + rB_;                                                                        \
        }                                                                                                                         \
        if (cmask & (1u << (3 * JJ))) {                                                                                           \
            double qA, qB;                                                                                                        \
            F2_SQ(erA, eiA, CcA, ScA, hq, dzq, mqrA, mqiA, qA)                                                                    \
            F2_SQ(erB, eiB, CcB, ScB, hq, dzq, mqrB, mqiB, qB)                                                                    \
            if (has_p) acc[20 + JJ] += qA + qB; else acc[JJ] += qA + qB;                                                          \
        }                                                                                                                         \
    }
                    double2 WaA, HaA, WaB, HaB, WbA, HbA, WbB, HbB; double La, Lb;
                    {
                        const double2 rf = s_rec[jfirst];
                        WaA = wtA[F2_OW(rf)]; HaA = htA[F2_OH(rf)]; WaB = wtB[F2_OW(rf)]; HaB = htB[F2_OH(rf)]; La = rf.x;
                        WbA = WaA; HbA = HaA; WbB = WaB; HbB = HaB; Lb = La;
                    }
                    switch (jj) {
                    case 0: F2_P1_NODE(0, WaA, HaA, WaB, HaB, La, WbA, HbA, WbB, HbB, Lb); jj = 1; if (jlast <= 1) break;
                    case 1: F2_P1_NODE(1, WbA, HbA, WbB, HbB, Lb, WaA, HaA, WaB, HaB, La); jj = 2; if (jlast <= 2) break;
                    case 2: F2_P1_NODE(2, WaA, HaA, WaB, HaB, La, WbA, HbA, WbB, HbB, Lb); jj = 3; if (jlast <= 3) break;
                    case 3: F2_P1_NODE(3, WbA, HbA, WbB, HbB, Lb, WaA, HaA, WaB, HaB, La); jj = 4; if (jlast <= 4) break;
                    case 4: F2_P1_NODE(4, WaA, HaA, WaB, HaB, La, WbA, HbA, WbB, HbB, Lb); jj = 5; if (jlast <= 5) break;
                    case 5: F2_P1_NODE(5, WbA, HbA, WbB, HbB, Lb, WaA, HaA, WaB, HaB, La); jj = 6; if (jlast <= 6) break;
                    case 6: F2_P1_NODE(6, WaA, HaA, WaB, HaB, La, WbA, HbA, WbB, HbB, Lb); jj = 7; if (jlast <= 7) break;
                    case 7: F2_P1_NODE(7, WbA, HbA, WbB, HbB, Lb, WaA, HaA, WaB, HaB, La); jj = 8; if (jlast <= 8) break;
                    case 8: F2_P1_NODE(8, WaA, HaA, WaB, HaB, La, WbA, HbA, WbB, HbB, Lb); jj = 9; if (jlast <= 9) break;
                    case 9: F2_P1_NODE(9, WbA, HbA, WbB, HbB, Lb, WaA, HaA, WaB, HaB, La); jj = 10;
                    }
#undef F2_P1_NODE
#undef F2_SQ
#undef F2_STEP_BIN
                }
            }
            // warp sum of the 30 accumulators through a padded shared-memory transpose, 8 values per round (fixed order)
            {
                double *tr = s_trans + warp * (F2_TRW * 33);
                const int row = lane & 7, part = lane >> 3;
#pragma unroll
                for (int rd = 0; rd < 4; rd++) {
                    if (!(rmask & (1u << rd))) continue;          // no active direction among these eight slots (per design)
#pragma unroll
                    for (int v = 0; v < F2_TRW; v++) tr[v * 33 + lane] = acc[rd * F2_TRW + v];
                    __syncwarp();
                    double sum = 0.0;
#pragma unroll
                    for (int x = 0; x < 8; x++) sum += tr[row * 33 + part * 8 + x];
                    sum += __shfl_xor_sync(0xffffffffu, sum, 8);
                    sum += __shfl_xor_sync(0xffffffffu, sum, 16);
                    if (lane < 8) s_wpart[(ch * nwarps + warp) * 32 + rd * F2_TRW + lane] = sum;
                    __syncwarp();
                }
            }
        }
        __syncthreads();
        for (int t = tid; t < nchunk * 32; t += T) {
            const int ch = t >> 5, l = t & 31;
            double s = 0.0;
            for (int wv = 0; wv < nwarps; wv++) s += s_wpart[(ch * nwarps + wv) * 32 + l];
            s_sums[par * sums_stride + t] = s;
        }
        if (CS > 1) {
            cluster.sync();
            for (int t = tid; t < nchunk * 32; t += T) {
                // every rank's partial is requested before the first one is used (a remote shared-memory read takes ~200
                // cycles); ranks beyond the cluster contribute an exact +0.0, so the sum keeps its order and value
                double s = 0.0;
#pragma unroll 1
                for (int r0 = 0; r0 < CS; r0 += 4) {
                    double v[4];
#pragma unroll
                    for (int r = 0; r < 4; r++) v[r] = (r0 + r < CS) ? cluster.map_shared_rank(s_sums, r0 + r)[par * sums_stride + t] : 0.0;
#pragma unroll
                    for (int r = 0; r < 4; r++) s += v[r];
                }
                s_tot[t] = s;
            }
        } else {
            __syncthreads();
            for (int t = tid; t < nchunk * 32; t += T) s_tot[t] = s_sums[par * sums_stride + t];
        }
        __syncthreads();

        // ================= linearised coefficients per node, member sums, B_drag ===================================
        for (int j = tid; j < Ns; j += T) {
            const int ch = j / CHUNK_NODES, jj = j - ch * CHUNK_NODES;
            const unsigned mk = ((unsigned)s_chunk[2 * ch] >> (3 * jj)) & 3u;
            // slot layout of the chunk (k_fused_plan): transverse-1 | transverse-2 | axial-when-both; axial alone sits in slot 0
            const double sA = s_tot[ch * 32 + jj], sB = s_tot[ch * 32 + 10 + jj], sC = s_tot[ch * 32 + 20 + jj];
            const double sq = (mk & 1u) ? ((mk & 2u) ? sC : sA) : 0.0, s1 = (mk & 2u) ? sA : 0.0, s2 = (mk & 2u) ? sB : 0.0;
            const bool circ = s_imem[IMEM_STRIDE * s_nodem[j] + 2] != 0;
            const double vq = sqrt(0.5 * sq);
            const double v1 = circ ? sqrt(0.5 * (s1 + s2)) : sqrt(0.5 * s1);
            const double v2 = circ ? v1 : sqrt(0.5 * s2);
            const double ls = n_ls[j], b1 = n_cd1[j] * v1, b2 = n_cd2[j] * v2;
            s_coef[0 * NsP + j] = n_cdq[j] * vq;
            s_coef[1 * NsP + j] = b1; s_coef[2 * NsP + j] = ls * b1;
            s_coef[3 * NsP + j] = b2; s_coef[4 * NsP + j] = ls * b2;
        }
        __syncthreads();
        for (int m = tid; m < Nm; m += T) {
            double bq = 0, b1 = 0, b1l = 0, b1ll = 0, b2 = 0, b2l = 0, b2ll = 0;
            for (int j = s_imem[IMEM_STRIDE * m]; j < s_imem[IMEM_STRIDE * m + 1]; j++) {
                const double ls = n_ls[j], q_ = s_coef[j], p1_ = s_coef[NsP + j], p2_ = s_coef[3 * NsP + j];
                bq += q_; b1 += p1_; b1l += p1_ * ls; b1ll += p1_ * ls * ls; b2 += p2_; b2l += p2_ * ls; b2ll += p2_ * ls * ls;
            }
            double *o = s_msum + m * 8;
            o[0] = bq; o[1] = b1; o[2] = b1l; o[3] = b1ll; o[4] = b2; o[5] = b2l; o[6] = b2ll;
        }
        __syncthreads();
        if (tid < 36) {
            const int a = tid / 6, b = tid % 6;
            double s = 0.0;
            for (int m = 0; m < Nm; m++) {
                const double *o = s_mem + m * MEM_STRIDE, *ms = s_msum + m * 8;
                const double vqa = a < 3 ? o[a] : o[9 + a - 3], vqb = b < 3 ? o[b] : o[9 + b - 3];
                const double v1a = a < 3 ? o[3 + a] : o[12 + a - 3], v1b = b < 3 ? o[3 + b] : o[12 + b - 3];
                const double v2a = a < 3 ? o[6 + a] : o[15 + a - 3], v2b = b < 3 ? o[6 + b] : o[15 + b - 3];
                const double u1a = a < 3 ? 0.0 : o[6 + a - 3], u1b = b < 3 ? 0.0 : o[6 + b - 3];
                const double u2a = a < 3 ? 0.0 : -o[3 + a - 3], u2b = b < 3 ? 0.0 : -o[3 + b - 3];
                s += ms[0] * vqa * vqb;
                s += ms[1] * v1a * v1b + ms[2] * (v1a * u1b + u1a * v1b) + ms[3] * u1a * u1b;
                s += ms[4] * v2a * v2b + ms[5] * (v2a * u2b + u2a * v2b) + ms[6] * u2a * u2b;
            }
            s_bmat[tid] = s_mat[36 + tid] + s;
            if (P.Bdrag_out && rank == 0) P.Bdrag_out[((size_t)d * Cs.nC + c) * 36 + tid] = s;
        }
        __syncthreads();
        if (FULL && P.lin_g && P.phase == 0 && rank == 0) {
            double *dst = P.lin_g + ((size_t)d * Cs.nC + c) * lin_stride;
#pragma unroll 1
            for (int t = tid; t < NCOEF * NsP; t += T) dst[t] = s_coef[t];
#pragma unroll 1
            for (int t = tid; t < 36; t += T) dst[NCOEF * NsP + t] = s_bmat[t];
        }
        }   // !secondary

        // ================= pass part 2: drag excitation of both bins (interleaved walk) ============================
        int conv_local = 1, nan_local = 0;
        const double *cq_ = s_coef, *c1_ = s_coef + NsP, *cl1_ = s_coef + 2 * NsP, *c2_ = s_coef + 3 * NsP, *cl2_ = s_coef + 4 * NsP;
        double brA[6], biA[6], brB[6], biB[6];
#pragma unroll
        for (int a = 0; a < 6; a++) { brA[a] = 0.0; biA[a] = 0.0; brB[a] = 0.0; biB[a] = 0.0; }
        {
            double2 eA = ok0 ? Eg[i0] : zero2, eB = ok1 ? Eg[i1] : zero2;                     // member 0, prefetched
            int zc = s_imem[4];
            double2 aA = Ag[(size_t)zc * nw + i0], aB = Ag[(size_t)zc * nw + i1];
            for (int m = 0; m < Nm; m++) {
                const double *o = s_mem + m * MEM_STRIDE;
                const double hq = o[18], h1 = o[19], h2 = o[20], dzq = o[2], dz1 = o[5], dz2 = o[8];
                const int j0 = s_imem[IMEM_STRIDE * m], j1 = s_imem[IMEM_STRIDE * m + 1];
                double erA = eA.x, eiA = eA.y, apA = aA.x, amA = aA.y, erB = eB.x, eiB = eB.y, apB = aB.x, amB = aB.y;
                if (m + 1 < Nm) {                                                              // next member's bases: in flight during this walk
                    zc = s_imem[IMEM_STRIDE * (m + 1) + 4];
                    eA = ok0 ? Eg[(size_t)(m + 1) * nw + i0] : zero2; eB = ok1 ? Eg[(size_t)(m + 1) * nw + i1] : zero2;
                    aA = Ag[(size_t)zc * nw + i0]; aB = Ag[(size_t)zc * nw + i1];
                }
                double AqrA = 0, AqiA = 0, A1rA = 0, A1iA = 0, A2rA = 0, A2iA = 0, L1rA = 0, L1iA = 0, L2rA = 0, L2iA = 0;
                double AqrB = 0, AqiB = 0, A1rB = 0, A1iB = 0, A2rB = 0, A2iB = 0, L1rB = 0, L1iB = 0, L2rB = 0, L2iB = 0;
#pragma unroll 2
                for (int j = j0; j < j1; j++) {
                    const double2 rj = s_rec[j];
                    const double2 WA = wtA[F2_OW(rj)], HA = htA[F2_OH(rj)], WB = wtB[F2_OW(rj)], HB = htB[F2_OH(rj)];
                    const double bq = cq_[j], b1 = c1_[j], lb1 = cl1_[j], b2 = c2_[j], lb2 = cl2_[j];
                    { const double tr = fma(erA, WA.x, -eiA * WA.y); eiA = fma(erA, WA.y, eiA * WA.x); erA = tr; }
                    { const double tr = fma(erB, WB.x, -eiB * WB.y); eiB = fma(erB, WB.y, eiB * WB.x); erB = tr; }
                    apA *= HA.x; amA *= HA.y; apB *= HB.x; amB *= HB.y;
                    const double CcA = apA + amA, ScA = apA - amA, CcB = apB + amB, ScB = apB - amB;
                    double crA, ciA, crB, ciB;
                    // a direction whose linearised coefficient is exactly zero adds exact zeros: skipped (same for every thread)
                    if (bq != 0.0) {
                        proj(erA, eiA, CcA, ScA, hq, dzq, crA, ciA); proj(erB, eiB, CcB, ScB, hq, dzq, crB, ciB);
                        AqrA = fma(bq, crA, AqrA); AqiA = fma(bq, ciA, AqiA); AqrB = fma(bq, crB, AqrB); AqiB = fma(bq, ciB, AqiB);
                    }
                    if (b1 != 0.0 || b2 != 0.0) {
                        proj(erA, eiA, CcA, ScA, h1, dz1, crA, ciA); proj(erB, eiB, CcB, ScB, h1, dz1, crB, ciB);
                        A1rA = fma(b1, crA, A1rA); A1iA = fma(b1, ciA, A1iA); L1rA = fma(lb1, crA, L1rA); L1iA = fma(lb1, ciA, L1iA);
                        A1rB = fma(b1, crB, A1rB); A1iB = fma(b1, ciB, A1iB); L1rB = fma(lb1, crB, L1rB); L1iB = fma(lb1, ciB, L1iB);
                        proj(erA, eiA, CcA, ScA, h2, dz2, crA, ciA); proj(erB, eiB, CcB, ScB, h2, dz2, crB, ciB);
                        A2rA = fma(b2, crA, A2rA); A2iA = fma(b2, ciA, A2iA); L2rA = fma(lb2, crA, L2rA); L2iA = fma(lb2, ciA, L2iA);
                        A2rB = fma(b2, crB, A2rB); A2iB = fma(b2, ciB, A2iB); L2rB = fma(lb2, crB, L2rB); L2iB = fma(lb2, ciB, L2iB);
                    }
                }
#pragma unroll
                for (int a = 0; a < 3; a++) {
                    brA[a] += o[a] * AqrA + o[3 + a] * A1rA + o[6 + a] * A2rA;
                    biA[a] += o[a] * AqiA + o[3 + a] * A1iA + o[6 + a] * A2iA;
                    brA[3 + a] += o[9 + a] * AqrA + o[12 + a] * A1rA + o[15 + a] * A2rA + o[6 + a] * L1rA - o[3 + a] * L2rA;
                    biA[3 + a] += o[9 + a] * AqiA + o[12 + a] * A1iA + o[15 + a] * A2iA + o[6 + a] * L1iA - o[3 + a] * L2iA;
                    brB[a] += o[a] * AqrB + o[3 + a] * A1rB + o[6 + a] * A2rB;
                    biB[a] += o[a] * AqiB + o[3 + a] * A1iB + o[6 + a] * A2iB;
                    brB[3 + a] += o[9 + a] * AqrB + o[12 + a] * A1rB + o[15 + a] * A2rB + o[6 + a] * L1rB - o[3 + a] * L2rB;
                    biB[3 + a] += o[9 + a] * AqiB + o[12 + a] * A1iB + o[15 + a] * A2iB + o[6 + a] * L1iB - o[3 + a] * L2iB;
                }
            }
        }
        // bin B's drag excitation waits in its own output slot (global, L2) while bin A is solved: the 6x6 system needs
        // every register
        if (ok1) {
#pragma unroll
            for (int a = 0; a < 6; a++) P.Xi_out[ogl + (size_t)a * nw + i1] = make_double2(brB[a], biB[a]);
        }
        // ================= impedance, solve, convergence, relaxation: bin A, then bin B =============================
#pragma unroll 1
        for (int bsel = 0; bsel < 2; bsel++) {
            const bool okb = bsel == 0 ? ok0 : ok1;
            if (!okb) continue;
            const int t = bsel == 0 ? t0 : t1, i = ibase + t;
            const double w = bsel == 0 ? w0 : w1;
            double br[6], bi[6];
            if (bsel == 0) {
#pragma unroll
                for (int a = 0; a < 6; a++) { br[a] = brA[a]; bi[a] = biA[a]; }
            } else {
#pragma unroll
                for (int a = 0; a < 6; a++) { const double2 v = P.Xi_out[ogl + (size_t)a * nw + i]; br[a] = v.x; bi[a] = v.y; }
            }
            if (FULL && P.Fdrag_out) {
#pragma unroll
                for (int a = 0; a < 6; a++) P.Fdrag_out[ogl + (size_t)a * nw + i] = make_double2(br[a], bi[a]);
            }
            double2 f0v[6];
#pragma unroll
            for (int a = 0; a < 6; a++) f0v[a] = P.F0g[ogl + (size_t)a * nw + i];          // in flight during the assembly
            double ar[6][6], ai[6][6];
            const double w2 = w * w;
            if (Aw) {
#pragma unroll
                for (int a = 0; a < 6; a++)
#pragma unroll
                    for (int b = 0; b < 6; b++) {
                        const double M = s_mat[6 * a + b] + Aw[(size_t)(6 * a + b) * nw + i];
                        const double B = s_bmat[6 * a + b] + Bw[(size_t)(6 * a + b) * nw + i];
                        ar[a][b] = fma(-w2, M, s_mat[72 + 6 * a + b]);
                        ai[a][b] = w * B;
                    }
            } else {
#pragma unroll
                for (int a = 0; a < 6; a++)
#pragma unroll
                    for (int b = 0; b < 6; b++) {
                        ar[a][b] = fma(-w2, s_mat[6 * a + b], s_mat[72 + 6 * a + b]);
                        ai[a][b] = w * s_bmat[6 * a + b];
                    }
            }
#pragma unroll
            for (int a = 0; a < 6; a++) { br[a] += f0v[a].x; bi[a] += f0v[a].y; }
            const bool ok = solve6(ar, ai, br, bi);
            if (!ok) nan_local |= RAFTK_FLAG_SINGULAR;
#pragma unroll
            for (int a = 0; a < 6; a++) {
                const double lr = s_xi[(2 * a) * nwl + t], li = s_xi[(2 * a + 1) * nwl + t];
                if (isnan(br[a]) || isnan(bi[a])) nan_local |= RAFTK_FLAG_NAN;
                if (!conv_ok(br[a] - lr, bi[a] - li, br[a], bi[a], P.tol)) conv_local = 0;
                s_xi[(2 * a) * nwl + t] = 0.2 * lr + 0.8 * br[a];
                s_xi[(2 * a + 1) * nwl + t] = 0.2 * li + 0.8 * bi[a];
                P.Xi_out[ogl + (size_t)a * nw + i] = make_double2(br[a], bi[a]);
                if (FULL && P.Xilast_out) P.Xilast_out[ogl + (size_t)a * nw + i] = make_double2(lr, li);
            }
        }
        passes++;
        // bit 0 = some bin not converged, bits 1.. = NaN / singular: one warp OR, one CTA barrier for all three flags
        int conv_all, nan_all;
        {
            const unsigned word = __reduce_or_sync(0xffffffffu, (unsigned)(conv_local ? 0 : 1) | ((unsigned)nan_local << 1));
            if (lane == 0) s_flw[warp] = (int)word;
            __syncthreads();
            unsigned all = 0;
#pragma unroll
            for (int wv = 0; wv < nwarps; wv++) all |= (unsigned)s_flw[wv];
            conv_all = !(all & 1u);
            nan_all = (int)(all >> 1) & (RAFTK_FLAG_NAN | RAFTK_FLAG_SINGULAR);
        }
        if (CS > 1) {
            if (tid == 0) { s_sums[par * sums_stride + nchunk * 32] = (double)conv_all; s_sums[par * sums_stride + nchunk * 32 + 1] = (double)nan_all; }
            cluster.sync();
            int ca = 1, na = 0;
#pragma unroll 1
            for (int r0 = 0; r0 < CS; r0 += 4) {
                double fc[4], fn[4];
#pragma unroll
                for (int r = 0; r < 4; r++) {                 // four ranks' flag words in flight at a time
                    const double *rem = cluster.map_shared_rank(s_sums, r0 + r < CS ? r0 + r : 0) + par * sums_stride + nchunk * 32;
                    fc[r] = rem[0]; fn[r] = rem[1];
                }
#pragma unroll
                for (int r = 0; r < 4; r++) { ca &= (int)fc[r]; na |= (int)fn[r]; }
            }
            conv_all = ca; nan_all = na;
        }
        par ^= 1;
        flags |= nan_all;
        if (nan_all & RAFTK_FLAG_NAN) break;
        if (conv_all) { converged = 1; break; }
    }
#undef F2_OW
#undef F2_OH
    if (P.status && rank == 0 && tid == 0) {
        int *st = P.status + ((size_t)d * Cs.nC + c) * 4;
        st[0] = secondary ? 0 : passes; st[1] = secondary ? 1 : converged; st[2] = flags; st[3] = secondary ? prim + 1 : 0;
    }
    if (P.n_peers > 1) {
        for (int t = tid; t < nloc; t += T) {
            const int i = f_begin + t;
#pragma unroll
            for (int a = 0; a < 6; a++) {
                const size_t o_ = ogl + (size_t)a * nw + i;
                const double2 v = P.Xi_out[o_];
#pragma unroll 1
                for (int pr = 0; pr < P.n_peers; pr++)
                    if (pr != P.peer_rank) P.peer_Xi[pr][o_] = v;
            }
        }
        if (rank == 0 && tid == 0) {
            const size_t so = ((size_t)d * Cs.nC + c) * 4;
#pragma unroll 1
            for (int pr = 0; pr < P.n_peers; pr++)
                if (pr != P.peer_rank && P.peer_status[pr]) {
                    int *st = P.peer_status[pr] + so;
                    st[0] = secondary ? 0 : passes; st[1] = secondary ? 1 : converged; st[2] = flags; st[3] = secondary ? prim + 1 : 0;
                }
        }
    }
    if (CS > 1) cluster.sync();
}
