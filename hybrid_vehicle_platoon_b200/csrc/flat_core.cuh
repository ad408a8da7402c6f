// flat_core.cuh -- per-vehicle local hybrid-MPC MIQP, one GPU THREAD per problem, written as a
// COMPACT flat state machine.
//
// Same mathematics as coop_core.cuh / miqp_core.cuh (problem: LocalMpcMld,
// fleet_decent_mld.py:61-208 on the pwa_gear model models.py:397-492; velocity-space node QPs,
// bounded-dual Goldfarb-Idnani with exact L1 slack elimination, depth-first branch and bound with
// relaxed-tail lower bounds).  The execution shape is what three rounds of ncu asked for:
//   * (r01a) one thread per problem with nested data-dependent loops: 5.8 of 32 lanes active;
//   * (r01b/c) fully unrolled / all-register variants: 6-9 k instructions of straight-line code,
//     55 % of the stall samples "no instruction" -- the kernel was bound by INSTRUCTION FETCH;
//   => this version keeps every loop rolled (#pragma unroll 1): the hot path (SELECT + STEP) is a
//      few hundred instructions and stays in the instruction cache; the per-thread vectors live in
//      a strided shared-memory slab (element e of lane l at slab[e*32 + l], conflict free);
//   * H^-1 is not rebuilt per node: moving between nodes of the depth-first search adds or removes
//     the input-cost term of one stage, a rank-1 change, so H^-1 follows by Sherman-Morrison
//     up/down-dates (O(N^2)) from the node it was last valid for;
//   * the solver is a state machine NEXT -> BUILD -> SELECT -> STEP; one trip() runs each block at
//     most once, in that order, so the 32 lanes of a warp (32 different problems) re-converge at
//     every block boundary; the kernel is persistent and a lane that finishes refills at once.
//
// Host + device (tests compile it with g++, ST = 1); the product only runs it inside local_miqp.cu.
#pragma once
#include <math.h>
#include <stdint.h>

#include "miqp_core.cuh"   // LocalParams, LocalResult, status codes, constraint type ids, HVP_HD

#if defined(__CUDACC__)
#define HVP_ROLL _Pragma("unroll 1")
#define HVP_FLAT_UNROLL _Pragma("unroll")
#else
#define HVP_ROLL
#define HVP_FLAT_UNROLL
#endif
#if defined(__CUDA_ARCH__)
#define HVP_LDG(p) __ldg(p)
#else
#define HVP_LDG(p) (*(p))
#endif

namespace hvp {

#if defined(__CUDA_ARCH__)
// The flat kernel runs one warp per CTA and its whole dynamic shared memory is the warp's work slab.
// Indexing this symbol (instead of a generic double*) tells the compiler the address space: LDS/STS with
// 32-bit address arithmetic instead of generic LD/ST with 64-bit pointer math (r01h ncu: 8.5 % of the
// issued instructions were generic loads and a quarter were IMAD/LEA address arithmetic).
extern __shared__ double hvp_flat_slab[];
#endif

// reciprocal to ~1 ulp without the slow paths of the IEEE division sequence
HVP_HD double hvp_rcp(double v) {
#if defined(__CUDA_ARCH__)
    // MUFU.RCP64H seed (20 bits, one instruction, no slow path) + two Newton steps (40, 80 bits): ~1 ulp
    double r;
    asm("rcp.approx.ftz.f64 %0, %1;" : "=d"(r) : "d"(v));
    r = r * (2.0 - v * r);
    r = r * (2.0 - v * r);
    return r;
#else
    return 1.0 / v;
#endif
}

#ifdef HVP_DEBUG_STATS
static long g_it[16], g_nodes[16], g_q[16], g_st[4], g_warm[8];
#endif
template <int N>
struct FlatLayout {
    static constexpr int TRI = N * (N + 1) / 2;
    static constexpr int O_HINV = 0;              // H^-1, full square (symmetric), row-major
    static constexpr int O_GINV = N * N;          // packed lower (N'H^-1N)^-1, slots a >= b
    static constexpr int O_X = O_GINV + TRI;
    static constexpr int O_LAM = O_X + N;
    static constexpr int O_YP = O_LAM + N;        // H^-1 n_p
    static constexpr int O_D = O_YP + N;          // d = N'yp (dead once r is known) ...
    static constexpr int O_WV = O_D;              // ... then w = n_p - N r and other scratch
    static constexpr int O_R = O_D + N;
    static constexpr int SIZE = O_R + N;          // doubles per thread (87 at N = 6: 10 warps / SM)
};

// Per-problem arrays that are indexed at run time.  They live OUTSIDE the solver object, in an object of their own
// that the caller owns: a run-time index into a member array keeps the compiler from promoting ANY member of
// the enclosing object to registers (r01j ncu: every scalar of the solver was re-loaded from local memory at the
// top of each block of the state machine -- long-scoreboard stalls on `L`, `act_lo`, `it`, `dual`, ...).
template <int N>
struct FlatCold {
    double gt[N], xstar[N], rlo[N + 1], rhi[N + 1], amax[N], amin[N];
    long long t_start;                  // device clock when the problem was picked up (time_limit_ns)
    // Sibling bounds (do_next): what the SOLVED parent of level l says about forcing v_l out of its relaxed value --
    // pf = the parent's optimum, pnz = curvature of its dual function along the bound row e_{l-1}, ptp / ptm = how far
    // the dual step may go before an active multiplier leaves [0, w] (row +e: regions below the relaxed v_l, row -e:
    // regions above).  pf = -inf: the level was created without solving its parent (first dive, adopted branch).
    double pf[N + 1], pnz[N + 1], ptp[N + 1], ptm[N + 1];
};

// ALG2 = the two refinements of the search that pay on a CPU and not on the GPU (measured, DESIGN.md 2.2): bounds on
// the siblings from the dual of their solved parent, and warm starts of first children from the parent's active set.
// They cut the work per solve by a third (10.4 -> 6.8 nodes, 50.6 -> 25.7 active-set steps at n = 10, N = 6) and the
// CPU port by the same; on the GPU the kernel is bound by instruction fetch and lane divergence, the extra code costs
// 10 % and fewer steps per node leave fewer lanes in step, so the CUDA kernels instantiate ALG2 = false.
// HINTS: compile the incumbent-hint entry (apply_hint) in.  A separate instantiation, because the kernel is bound by
// instruction fetch: 150 instructions that never run still cost the un-hinted launch 5 % (r02 measurement).
template <int N, int ST, bool ALG2 = false, bool HINTS = false>
struct FlatSolver {
    using LY = FlatLayout<N>;
    enum : int { S_NEXT = 0, S_BUILD, S_SELECT, S_STEP, S_DONE };
    // Interval-hull tightening of the unfixed stages (hull()).  It pays in the compiled-MPC kernel (pm_kernel.cu) but
    // not here (N = 6: same node count, more work per node), so it is compiled OUT: the kernel's code must stay
    // inside the 32 KB instruction cache level (r01l ncu: 'no instruction' was the second largest stall reason).
    static constexpr bool kHull = false;

    double* W;
    const LocalParams* P;
    const double* xf_;                  // soft-row data is read from the caller's arrays
    const double* xb_;
    double* best_;                      // incumbent velocities go straight to the output trajectory
    FlatCold<N>* C;                     // cold per-problem arrays (touched once per node): thread-local memory
    double p0, v0, pc, inv_m, a_lo, a_hi, c_lo, c_hi, hw1, hw2, hd, ct;
    bool has_sf, has_sb;
    // soft-row right-hand sides sf(j), sb(j), j = 1..N-1, read ONCE per problem.  Indexed with compile-time
    // constants only (a run-time index would push the whole solver object back into local memory).
    double sfv[N], sbv[N];
    // branch and bound
    int state, lev, L, nodes, iters, it;
    double inc;
    uint64_t modes_pk, best_modes, cand_pk, built_pk;   // 3 bits / stage; 7 candidate bits / level
    int built_L;                                        // H^-1 currently holds stages 0..built_L-1 of built_pk
    bool trouble, limit, timeout;
    bool notrack;                                       // no reference term: only leaves are solved
    bool dive;                                          // first descent: path nodes are not solved, only the leaf
    bool hinted;                                        // the node being solved is the caller's hinted leaf
    int hint_c0;
    bool fresh;                                         // the slab still holds the solved parent of level `lev`
#ifdef HVP_DEBUG_STATS
    bool was_warm = false;
#endif
    bool slab_ok;                                       // ... and nothing has been built since (warm start of its first child)
    // active set
    int q;
    uint64_t act_lo, act_hi;                            // slot bytes (act_raw), 8 bits each
    uint32_t satf, satb;
    // constraint being added
    int pcode, pkind, pj;                               // pcode: p's slot byte once it is added (act_raw)
    double psgn, pcoef, nHn, lam_p, cp;
    double dual;                                         // value of the node's dual function (lower bound)
    bool p_soft;

    int lane_;                          // lane of this problem within the warp (device)
    HVP_HD double& w(int off, int i) const {
#if defined(__CUDA_ARCH__)
        return hvp_flat_slab[(off + i) * ST + lane_];
#else
        return W[(size_t)(off + i) * ST];
#endif
    }
    HVP_HD static int tri(int a, int b) { return a * (a + 1) / 2 + b; }          // a >= b
    // max / min of operands that are never NaN (parameters, merged bounds): a compare and two selects instead of the
    // NaN handling of fmax / fmin
    HVP_HD static double nmax(double a, double b) { return a > b ? a : b; }
    HVP_HD static double nmin(double a, double b) { return a < b ? a : b; }
    HVP_HD double ra(int rg) const { return rg < 4 ? a_lo : a_hi; }
    HVP_HD double rc(int rg) const { return rg < 4 ? c_lo : c_hi; }
    HVP_HD double rb(int rg) const { return P->bgear[rg] * inv_m; }
    HVP_HD static int mode_of(uint64_t pk, int k) { return (int)((pk >> (3 * k)) & 7u); }
    HVP_HD int mode(int k) const { return mode_of(modes_pk, k); }
    HVP_HD void set_mode(int k, int rg) { modes_pk = (modes_pk & ~(7ull << (3 * k))) | ((uint64_t)rg << (3 * k)); }
    HVP_HD int cand(int lv) const { return (int)((cand_pk >> (7 * lv)) & 0x7fu); }
    HVP_HD void set_cand(int lv, int v) { cand_pk = (cand_pk & ~(0x7full << (7 * lv))) | ((uint64_t)v << (7 * lv)); }
    // Slot a's row is one byte, decoded when the row enters the active set so that the products over the active set
    // read it with masks only: bits 0-3 = stage j, bit 4 = the row enters with sign -1 (the sign includes a soft row's
    // orientation at the time it became active; it cannot flip while active), bits 5-7 = row class (R_*), which fixes
    // the row's shape and, for input-limit rows, its difference coefficient a_r (the region of stage j is fixed for the
    // whole node).  A (class, sign, stage) byte identifies the row: UB / LB, ACC / DEC, ... differ in the sign bit.
    enum : int { R_BOUND = 0, R_ACC, R_IN_LO, R_IN_HI, R_POS, R_SF, R_SB };
    // row class of each constraint type (miqp_core.cuh T_*), 4 bits per type; input-limit rows add 1 in regions >= 4
    static constexpr uint64_t kClassOfType = 0x6544221100ull;
    // q <= N (a row dependent on the active set is never added), so act_hi is only used at N = 9
    HVP_HD int act_raw(int a) const { return (int)((((N <= 8 || a < 8) ? act_lo >> (8 * a) : act_hi >> (8 * (a - 8)))) & 0xffu); }
    HVP_HD static bool slot_soft(int b) { return b >= (R_SF << 5); }
    HVP_HD double slot_coef(int b) const {           // difference coefficient: a_r of the stage for input-limit rows
        const int cls = b >> 5;
        return cls == R_IN_LO ? a_lo : (cls == R_IN_HI ? a_hi : 1.0);
    }
    // the slot bytes in order, from a copy of act_lo / act_hi shifted by one slot per call (constant shifts)
    struct SlotIter {
        uint64_t lo, hi;
        HVP_HD int next() {
            const int b = (int)(lo & 0xffu);
            lo >>= 8;
            if (N > 8) { lo |= hi << 56; hi >>= 8; }
            return b;
        }
    };
    HVP_HD SlotIter slots() const { return SlotIter{act_lo, act_hi}; }
    HVP_HD void set_act(int a, int id) {
        if (N <= 8 || a < 8) act_lo = (act_lo & ~(0xffull << (8 * a))) | ((uint64_t)id << (8 * a));
        else act_hi = (act_hi & ~(0xffull << (8 * (a - 8)))) | ((uint64_t)id << (8 * (a - 8)));
    }
    HVP_HD double Hoff(int j) const { return hw1 * (double)(N - 1 - j) + hw2; }
    HVP_HD double Hdiag(int j) const { return hw1 * (double)(N - 1 - j) + hd; }
    HVP_HD double sf(int j) const { return HVP_LDG(xf_ + j + 1) - P->d_safe - pc; }       // rows PS_j <= sf(j)
    HVP_HD double sb(int j) const { return HVP_LDG(xb_ + j + 1) + P->d_safe - pc; }       // rows PS_j >= sb(j)

    // -------------------------------------------------------------------------------------
    HVP_HD void setup(double* W_, const LocalParams* P_, int flags, double mass, const double* x0,
                      const double* xf, const double* xb, const double* xl, double* best_out, FlatCold<N>* cold) {
        W = W_; P = P_; xf_ = xf; xb_ = xb; best_ = best_out; C = cold;
        p0 = x0[0]; v0 = x0[1]; pc = p0 + v0;
        inv_m = hvp_rcp(mass);
        a_lo = 1.0 - P->c1 * inv_m; a_hi = 1.0 - P->c2 * inv_m;
        c_lo = -P->mug; c_hi = -P->mug - P->dfr * inv_m;
        const bool is_front = flags & 1, is_leader = flags & 2, is_trailer = flags & 4;
        const bool tf = !is_front && !is_leader, tb = !is_trailer && !is_leader, tl = is_leader;
        const double wp = P->qxp, wvv = P->qxv, t0 = P->t0, d0 = P->d0;
        const int np1 = N + 1;
        const double nterm = (tf ? 1.0 : 0.0) + (tb ? 1.0 : 0.0) + (tl ? 1.0 : 0.0);
        hw1 = 2.0 * wp * nterm;
        hw2 = 2.0 * wp * (tf ? t0 : 0.0);
        hd = 2.0 * wp * (tf ? t0 * t0 : 0.0) + 2.0 * wvv * nterm;
        HVP_ROLL
        for (int j = 0; j < N; ++j) C->gt[j] = 0.0;
        ct = 0.0;
        HVP_ROLL
        for (int kind = 0; kind < 3; ++kind) {
            const double* ref = kind == 0 ? xf : (kind == 1 ? xb : xl);
            const bool on = kind == 0 ? tf : (kind == 1 ? tb : tl);
            if (!on) continue;
            const double tau = kind == 0 ? t0 : 0.0;
            double suffix = 0.0;
            HVP_ROLL
            for (int k = N; k >= 0; --k) {
                const double pk = ref[k], vk = ref[np1 + k];
                const double Pk = (kind == 0) ? (pk - d0) : (kind == 1) ? (pk + t0 * vk + d0) : pk;
                if (k >= 1) {
                    const double rho = pc - Pk;
                    C->gt[k - 1] += 2.0 * wp * (suffix + tau * rho) - 2.0 * wvv * vk;
                    ct += wp * rho * rho + wvv * vk * vk;
                    suffix += rho;
                } else {
                    const double e0 = p0 + tau * v0 - Pk, e1 = v0 - vk;
                    ct += wp * e0 * e0 + wvv * e1 * e1;
                }
            }
        }
        has_sf = !is_front; has_sb = !is_trailer;
        const double ww = P->w, ds = P->d_safe;
        if (has_sf) {
            const double s0 = p0 - (xf[0] - ds), s1 = pc - (xf[1] - ds);
            ct += ww * (s0 > 0 ? s0 : 0.0) + ww * (s1 > 0 ? s1 : 0.0);
        }
        if (has_sb) {
            const double s0 = (xb[0] + ds) - p0, s1 = (xb[1] + ds) - pc;
            ct += ww * (s0 > 0 ? s0 : 0.0) + ww * (s1 > 0 ? s1 : 0.0);
        }
        HVP_FLAT_UNROLL
        for (int j = 1; j < N; ++j) {
            sfv[j] = has_sf ? sf(j) : 0.0;
            sbv[j] = has_sb ? sb(j) : 0.0;
        }
        sfv[0] = sbv[0] = 0.0;
        // ---- H^-1 of the pure tracking Hessian (no stage fixed): one of three matrices the host inverted ----
        // Without a reference term (a front vehicle that is also the trailer and not the leader) the Hessian is the
        // input cost of the fixed stages alone: singular at every node that leaves a stage free.  Such a problem is
        // searched over its leaves only (do_next), and each leaf inverts its own Hessian (leaf_inverse).
        notrack = nterm < 0.5;
        if (!notrack) {
            const double* h0 = P->h0inv[tf ? (tb ? 2 : 1) : 0];
            HVP_ROLL
            for (int e = 0; e < N * N; ++e) w(LY::O_HINV, e) = h0[e];
        }
        built_L = 0; built_pk = 0;
        // ---- start of the search ----
        iters = 0; nodes = 0; it = 0; modes_pk = 0; best_modes = 0; cand_pk = 0;
        inc = HUGE_VAL; trouble = limit = timeout = false; lev = 0; dive = P->dive != 0; fresh = false; slab_ok = false;
        hinted = false;
        if (P->time_limit_ns > 0) C->t_start = hvp_now_ns();
        if (ALG2) C->pf[0] = -HUGE_VAL;
        int c0 = 0;
        HVP_ROLL
        for (int rg = 0; rg < NREG; ++rg)
            if (v0 >= P->edge[rg] && v0 <= P->edge[rg + 1]) c0 |= (1 << rg);
        set_cand(0, c0);
        C->xstar[0] = v0; C->rlo[0] = v0; C->rhi[0] = v0;
        state = S_NEXT;
    }

    // ---- incumbent hint (include/hvp.h: modes_hint) ----------------------------------------------------------------
    // In a closed loop the previous timestep's optimal region sequence, shifted by one stage, is almost always a
    // feasible leaf of this timestep's tree and very often the optimal one.  Solving that ONE leaf first gives the
    // search an incumbent before any relaxation is solved: the first dive (two QPs whose only purpose is an incumbent)
    // is skipped and the root relaxations are pruned by their dual bounds.  The hint is advice, never trusted: a
    // sequence that is out of range, starts in a region that does not contain v0 or turns out infeasible is dropped and
    // the search runs as if no hint had been given; either way the search that follows proves the optimum.
    HVP_HD void apply_hint(const int32_t* h) {
        // descend along the hinted sequence exactly as the first dive would: regions fixed, intervals propagated,
        // siblings left on the depth-first stack, NOTHING solved on the way -- only the leaf
        const double eps = 1e-9;
        const int c0 = cand(0);
        bool ok = true;
        HVP_ROLL
        for (int lv = 0; lv < N && ok; ++lv) {
            const int rg = h[lv];
            int cn = c0;
            if (lv > 0) {
                cn = 0;
                HVP_ROLL
                for (int c = 0; c < NREG; ++c)
                    if (P->edge[c] <= C->rhi[lv] && P->edge[c + 1] >= C->rlo[lv]) cn |= (1 << c);
            }
            if (rg < 0 || rg >= NREG || !((cn >> rg) & 1)) { ok = false; break; }
            set_mode(lv, rg);
            set_cand(lv, cn & ~(1 << rg));
            const double jlo = fmax(C->rlo[lv], P->edge[rg]), jhi = fmin(C->rhi[lv], P->edge[rg + 1]);
            double nlo = fmax(ra(rg) * jlo + rc(rg) + rb(rg) * P->umin, jlo + P->a_dec + lv * P->tight);
            double nhi = fmin(ra(rg) * jhi + rc(rg) + rb(rg) * P->umax, jhi + P->a_acc - lv * P->tight);
            nlo = fmax(nlo, P->vmin); nhi = fmin(nhi, P->vmax);
            if (jlo > jhi + eps || nlo > nhi + eps) { ok = false; break; }
            if (lv + 1 < N) { C->rlo[lv + 1] = nlo - eps; C->rhi[lv + 1] = nhi + eps; C->xstar[lv + 1] = v0; }
        }
        if (!ok || pc > P->pmax + eps || pc < P->pmin - eps) { unhint(c0); return; }
        hint_c0 = c0;
        lev = N - 1;
        L = N;
        hinted = true;
        state = S_BUILD;
    }
    HVP_HD void unhint(int c0) {           // back to the untouched start of the search
        modes_pk = 0; cand_pk = 0;
        set_cand(0, c0);
        lev = 0;
        state = S_NEXT;
    }

    // ---- sub-tree adoption (tail of a launch: idle lanes of the warp take open branches of a busy lane) -------
    // Shallowest level of the depth-first stack that still has untried regions, and how many are open in total.
    // Valid in state S_NEXT (levels above `lev` are exhausted there).
    HVP_HD bool open_level(int& l, int& cb, int& total) const {
        l = -1; cb = 0; total = 0;
        HVP_ROLL
        for (int lv = 0; lv <= lev; ++lv) {
            const int c = cand(lv);
            if (c && l < 0) { l = lv; cb = c; }
            total += __builtin_popcount((unsigned)c);
        }
        return l >= 0;
    }
    // After setup() of the SAME problem: follow the donor's region prefix (levels 0..l-1, interval propagation as in
    // do_next, nothing is solved) and search only region `c` at level l, starting from the donor's incumbent.
    HVP_HD void adopt_prefix(uint64_t donor_modes, int l, int c, double donor_inc) {
        const double eps = 1e-9;
        HVP_ROLL
        for (int lv = 0; lv < l; ++lv) {
            const int rg = mode_of(donor_modes, lv);
            set_mode(lv, rg);
            set_cand(lv, 0);
            const double jlo = fmax(C->rlo[lv], P->edge[rg]), jhi = fmin(C->rhi[lv], P->edge[rg + 1]);
            double nlo = fmax(ra(rg) * jlo + rc(rg) + rb(rg) * P->umin, jlo + P->a_dec + lv * P->tight);
            double nhi = fmin(ra(rg) * jhi + rc(rg) + rb(rg) * P->umax, jhi + P->a_acc - lv * P->tight);
            nlo = fmax(nlo, P->vmin); nhi = fmin(nhi, P->vmax);
            C->rlo[lv + 1] = nlo - eps; C->rhi[lv + 1] = nhi + eps;
            C->xstar[lv + 1] = v0;
            if (ALG2) C->pf[lv + 1] = -HUGE_VAL;
        }
        fresh = false; slab_ok = false;
        set_cand(l, 1 << c);
        lev = l;
        inc = donor_inc;
        dive = false;
        state = S_NEXT;
    }

    // ---- NEXT: next node of the depth-first search (or finished) --------------------------
    // Dual information of the node that has just been solved (the parent of level `lev`), taken while its active
    // set is still in the slab: the first step of the dual active-set method on a child that forces v_lev into a
    // region away from the relaxed value, WITHOUT building the child.  For the bound row n = +-e_{lev-1}:
    // yp = H^-1 n, d = N'yp, r = Ginv d, nz = n'yp - d'r; the dual function along the step is f + t*viol - t^2 nz / 2
    // for 0 <= t <= tmax (ratio tests).  Every child adds cost and rows to the parent, so this bounds it from below.
    HVP_HD void parent_info() {
        const double ww = P->w, INF = HUGE_VAL;
        const int pj0 = lev - 1;
        HVP_ROLL
        for (int i = 0; i < N; ++i) w(LY::O_YP, i) = w(LY::O_HINV, pj0 * N + i);
        const double nHn0 = w(LY::O_HINV, pj0 * N + pj0);
        SlotIter si = slots();
        HVP_ROLL
        for (int a = 0; a < q; ++a) w(LY::O_D, a) = slot_dot(si.next(), LY::O_YP);
        double nz = nHn0, tp = INF, tm = INF;
        HVP_ROLL
        for (int a = 0; a < q; ++a) {
            double s = 0.0;
            int gi = tri(a, 0);
            HVP_ROLL
            for (int b = 0; b <= a; ++b) s += w(LY::O_GINV, gi + b) * w(LY::O_D, b);
            gi += 2 * a + 1;
            HVP_ROLL
            for (int b = a + 1; b < q; ++b) { s += w(LY::O_GINV, gi) * w(LY::O_D, b); gi += b + 1; }
            nz -= s * w(LY::O_D, a);
            const double la = w(LY::O_LAM, a);
            const bool soft = slot_soft(act_raw(a));
            if (s > 1e-14) {
                const double is = hvp_rcp(s);
                tp = fmin(tp, la * is);
                if (soft) tm = fmin(tm, (ww - la) * is);
            } else if (s < -1e-14) {
                const double is = hvp_rcp(-s);
                tm = fmin(tm, la * is);
                if (soft) tp = fmin(tp, (ww - la) * is);
            }
        }
        if (q == N || !(nz > 1e-11 * nHn0)) nz = 0.0;          // dependent row: the dual is linear along the step
        C->pnz[lev] = nz; C->ptp[lev] = fmax(tp, 0.0); C->ptm[lev] = fmax(tm, 0.0);
    }

    HVP_HD void do_next() {
        const double eps = 1e-9;
        if (ALG2 && fresh) { parent_info(); fresh = false; }
        for (;;) {
            int cset = cand(lev);
            if (cset == 0) {
                if (lev == 0) { state = S_DONE; return; }
                --lev;
                continue;
            }
            int rg = -1; double bd = HUGE_VAL;
            const double xs = C->xstar[lev];
            HVP_ROLL
            for (int c = 0; c < NREG; ++c) {
                if (!((cset >> c) & 1)) continue;
                const double lo = P->edge[c], hi = P->edge[c + 1];
                const double dist = xs < lo ? lo - xs : (xs > hi ? xs - hi : 0.0);
                if (dist < bd) { bd = dist; rg = c; }
            }
            set_cand(lev, cset & ~(1 << rg));
            const double pf = ALG2 ? C->pf[lev] : -HUGE_VAL;
            if (ALG2 && bd > 0.0 && inc < HUGE_VAL && pf > -HUGE_VAL && P->sibling_bound) {
                // sibling bound from the solved parent (parent_info): cheaper than building the child to find out
                const double nz = C->pnz[lev];
                const double tmax = (xs > P->edge[rg + 1]) ? C->ptp[lev] : C->ptm[lev];
                const double t = (nz > 0.0) ? fmin(bd * hvp_rcp(nz), tmax) : tmax;
                const double bound = (t < HUGE_VAL) ? pf + t * bd - 0.5 * t * t * nz : HUGE_VAL;
                if (bound > inc) continue;
            }
            set_mode(lev, rg);
            const double jlo = fmax(C->rlo[lev], P->edge[rg]), jhi = fmin(C->rhi[lev], P->edge[rg + 1]);
            if (jlo > jhi + eps) continue;
            double nlo = fmax(ra(rg) * jlo + rc(rg) + rb(rg) * P->umin, jlo + P->a_dec + lev * P->tight);
            double nhi = fmin(ra(rg) * jhi + rc(rg) + rb(rg) * P->umax, jhi + P->a_acc - lev * P->tight);
            nlo = fmax(nlo, P->vmin); nhi = fmin(nhi, P->vmax);
            if (nlo > nhi + eps) continue;
            if (pc > P->pmax + eps || pc < P->pmin - eps) continue;
            C->rlo[lev + 1] = nlo - eps; C->rhi[lev + 1] = nhi + eps;
            L = lev + 1;
            if (((dive && nodes >= 1) || notrack) && L < N) {
                // First descent: no incumbent exists yet, so the relaxations along the path could not
                // prune anything -- they only guide the choice of region.  Keep following the last
                // relaxed trajectory and solve the LEAF directly; its objective is the first incumbent.
                // (notrack: every descent, as the oracle enumerates the leaves; no relaxation is solved.)
                ++lev;
                C->xstar[lev] = notrack ? C->xstar[lev - 1] : w(LY::O_X, lev - 1);
                if (ALG2) C->pf[lev] = -HUGE_VAL;        // no solved parent: no sibling bound at this level
                int cn = 0;
                HVP_ROLL
                for (int c = 0; c < NREG; ++c)
                    if (P->edge[c] <= C->rhi[lev] && P->edge[c + 1] >= C->rlo[lev]) cn |= (1 << c);
                set_cand(lev, cn);
                continue;
            }
            if (kHull) hull();
            state = S_BUILD;
            return;
        }
    }

    // Interval reachability of the stages that are not fixed yet: hull over the PWA regions of the
    // velocity interval and of the acceleration the traction / braking allows, stage by stage.  Every
    // completion of the node's region prefix satisfies these bounds, so the relaxation may impose them.
    HVP_HD void hull() {
        const double eps = 1e-9;
        double lo = C->rlo[L], hi = C->rhi[L];
        HVP_ROLL
        for (int s = L; s < N; ++s) {
            double nlo = HUGE_VAL, nhi = -HUGE_VAL, dmax = -HUGE_VAL, dmin = HUGE_VAL;
            HVP_ROLL
            for (int r = 0; r < NREG; ++r) {
                const double jlo = fmax(lo, P->edge[r]), jhi = fmin(hi, P->edge[r + 1]);
                if (jlo > jhi + eps) continue;
                const double a = ra(r), b = rb(r), c = rc(r);
                nlo = fmin(nlo, a * jlo + c + b * P->umin);
                nhi = fmax(nhi, a * jhi + c + b * P->umax);
                dmax = fmax(dmax, (a - 1.0) * jlo + c + b * P->umax);
                dmin = fmin(dmin, (a - 1.0) * jhi + c + b * P->umin);
            }
            const double acc = P->a_acc - s * P->tight, dec = P->a_dec + s * P->tight;
            C->amax[s] = fmin(dmax + eps, acc); C->amin[s] = fmax(dmin - eps, dec);
            nlo = fmax(fmax(nlo, lo + dec), P->vmin); nhi = fmin(fmin(nhi, hi + acc), P->vmax);
            lo = nlo - eps; hi = nhi + eps;
            C->rlo[s + 1] = lo; C->rhi[s + 1] = hi;
        }
    }

    HVP_HD void node_done(int st, double obj) {
        iters += it;
        ++nodes;
#ifdef HVP_DEBUG_STATS
        g_it[L] += it; g_nodes[L] += 1; g_q[L] += q; g_st[st] += 1;
        if (was_warm) { g_warm[3] += it; } else { g_warm[4] += it; g_warm[5] += 1; } was_warm = false;
#endif
        state = S_NEXT;
        if (HINTS && hinted) {
            hinted = false;
            if (st != 0) { --nodes; unhint(hint_c0); return; }   // infeasible hinted leaf: as if there had been no hint
            HVP_ROLL
            for (int lv = 1; lv < N; ++lv) C->xstar[lv] = w(LY::O_X, lv - 1);   // sibling order: distance to the leaf
        }
        if (st != 0 || L == N) dive = false;
        if (st == 2) { trouble = true; return; }
        if (st == 1) return;
        if (inc < HUGE_VAL && !(obj < hvp_cut(inc, P->mip_gap))) return;              // bound
        if (L == N) {                                                                // leaf
            inc = obj; best_modes = modes_pk;
            HVP_ROLL
            for (int j = 0; j < N; ++j) best_[j] = w(LY::O_X, j);
            return;
        }
        if (P->max_nodes > 0 && nodes >= P->max_nodes) { limit = true; state = S_DONE; return; }
        if (P->time_limit_ns > 0 && hvp_now_ns() - C->t_start > P->time_limit_ns) { timeout = true; state = S_DONE; return; }
        ++lev;
        C->xstar[lev] = w(LY::O_X, lev - 1);                                             // relaxed v_lev
        if (ALG2) { C->pf[lev] = fmin(obj, dual); fresh = true; slab_ok = true; }
        int cn = 0;
        HVP_ROLL
        for (int c = 0; c < NREG; ++c)
            if (P->edge[c] <= C->rhi[lev] && P->edge[c + 1] >= C->rlo[lev]) cn |= (1 << c);
        set_cand(lev, cn);
    }

    // H <- H + s * 2*qu * e e'  with  e = (e_k - a e_{k-1})/b  (stage k, region rg):
    // Sherman-Morrison on the stored H^-1;  s = +1 adds the stage's input cost, -1 removes it.
    HVP_HD double rank1(int k, int rg, double s) {
        const double ib = hvp_rcp(rb(rg)), ea = (k >= 1) ? -ra(rg) * ib : 0.0;
        double ev = 0.0;                                   // e' H^-1 e
        HVP_ROLL
        for (int i = 0; i < N; ++i) {
            double v = ib * w(LY::O_HINV, i * N + k);
            if (k >= 1) v += ea * w(LY::O_HINV, i * N + k - 1);
            w(LY::O_WV, i) = v;                            // v = H^-1 e
        }
        ev = ib * w(LY::O_WV, k) + ((k >= 1) ? ea * w(LY::O_WV, k - 1) : 0.0);
        const double den = hvp_rcp(1.0 / (2.0 * P->qu) * s + ev);     // (1/(s*2qu) + e'H^-1e)^-1, s = +-1
        double vr[N];                                      // v in registers: the inner loop has a compile-time trip count
        HVP_FLAT_UNROLL
        for (int j = 0; j < N; ++j) vr[j] = w(LY::O_WV, j);
        HVP_ROLL
        for (int i = 0; i < N; ++i) {
            const double vi = w(LY::O_WV, i) * den;
            HVP_FLAT_UNROLL
            for (int j = 0; j < N; ++j) w(LY::O_HINV, i * N + j) -= vi * vr[j];
        }
        return den;                                        // H'^-1 = H^-1 - den v v', v left in O_WV
    }

    // H^-1 of a leaf of a problem without reference terms (notrack): H = sum over the stages of the input cost
    // 2 qu e e', e = (e_k - a e_{k-1})/b, tridiagonal and positive definite once every stage is fixed;
    // in-place Gauss-Jordan (no pivoting needed)
    HVP_HD void leaf_inverse() {
        const double qu2 = 2.0 * P->qu;
        HVP_ROLL
        for (int e = 0; e < N * N; ++e) w(LY::O_HINV, e) = 0.0;
        HVP_ROLL
        for (int k = 0; k < N; ++k) {
            const int rg = mode(k);
            const double ib = hvp_rcp(rb(rg));
            w(LY::O_HINV, k * N + k) += qu2 * ib * ib;
            if (k >= 1) {
                const double ea = -ra(rg) * ib;
                w(LY::O_HINV, (k - 1) * N + k - 1) += qu2 * ea * ea;
                w(LY::O_HINV, k * N + k - 1) += qu2 * ea * ib;
                w(LY::O_HINV, (k - 1) * N + k) += qu2 * ea * ib;
            }
        }
        HVP_ROLL
        for (int k = 0; k < N; ++k) {
            const double pinv = hvp_rcp(w(LY::O_HINV, k * N + k));
            HVP_ROLL
            for (int j = 0; j < N; ++j) w(LY::O_HINV, k * N + j) *= pinv;
            w(LY::O_HINV, k * N + k) = pinv;
            HVP_ROLL
            for (int i = 0; i < N; ++i) {
                if (i == k) continue;
                const double f = w(LY::O_HINV, i * N + k);
                HVP_ROLL
                for (int j = 0; j < N; ++j)
                    w(LY::O_HINV, i * N + j) = (j == k) ? -f * pinv : w(LY::O_HINV, i * N + j) - f * w(LY::O_HINV, k * N + j);
            }
        }
    }

    // ---- BUILD: bring H^-1 to this node, gradient, unconstrained minimiser -----------------
    HVP_HD void do_build() {
        const double qu = P->qu, ww = P->w;
        // common prefix of the stages H^-1 currently contains and the stages this node fixes
        int c = 0;
        while (c < built_L && c < L && mode_of(built_pk, c) == mode(c)) ++c;
        // WARM START.  The slab still holds the optimum of the node's PARENT (x*, its active rows, their multipliers
        // and (N'H^-1N)^-1) when this is the first child built after the parent was solved.  The child adds one
        // rank-1 term to H (the input cost of stage L-1), so instead of re-adding the parent's ~N-1 active rows one
        // dual step at a time: update (N'H^-1N)^-1 by Sherman-Morrison, move to the minimiser on the SAME rows, and
        // keep that as the starting S-pair if every multiplier stays admissible (otherwise: the cold start below).
        const bool warm = ALG2 && slab_ok && P->warm && L == built_L + 1 && c == built_L && (satf | satb) == 0u && q > 0;
        slab_ok = false;
        if (warm) {
            const double den = rank1(L - 1, mode(L - 1), 1.0);              // v = H^-1 e in O_WV
            SlotIter si = slots();
            HVP_ROLL
            for (int a = 0; a < q; ++a) w(LY::O_R, a) = slot_dot(si.next(), LY::O_WV);   // z = N'v
            double zr = 0.0;
            HVP_ROLL
            for (int a = 0; a < q; ++a) {                                    // r = Ginv z  (into O_YP)
                double s = 0.0;
                int gi = tri(a, 0);
                HVP_ROLL
                for (int b = 0; b <= a; ++b) s += w(LY::O_GINV, gi + b) * w(LY::O_R, b);
                gi += 2 * a + 1;
                HVP_ROLL
                for (int b = a + 1; b < q; ++b) { s += w(LY::O_GINV, gi) * w(LY::O_R, b); gi += b + 1; }
                w(LY::O_YP, a) = s;
                zr += s * w(LY::O_R, a);
            }
            const double alpha = den * hvp_rcp(1.0 - den * zr);              // (G - den zz')^-1 = Ginv + alpha rr'
            HVP_ROLL
            for (int a = 0; a < q; ++a) {
                const double ra_ = alpha * w(LY::O_YP, a);
                HVP_ROLL
                for (int b = 0; b <= a; ++b) w(LY::O_GINV, tri(a, b)) += ra_ * w(LY::O_YP, b);
            }
        } else if (notrack) {
            leaf_inverse();
        } else {
            HVP_ROLL
            for (int k = built_L - 1; k >= c; --k) rank1(k, mode_of(built_pk, k), -1.0);
            HVP_ROLL
            for (int k = c; k < L; ++k) rank1(k, mode(k), 1.0);
        }
        built_L = L; built_pk = modes_pk;
        // gradient g = gt + input-cost terms (into O_D), then x = -H^-1 g
        HVP_ROLL
        for (int i = 0; i < N; ++i) w(LY::O_D, i) = C->gt[i];
        dual = ct;
        HVP_ROLL
        for (int k = 0; k < L; ++k) {
            const int rg = mode(k);
            const double ib = hvp_rcp(rb(rg)), ea = -ra(rg) * ib;
            const double kc = (k == 0) ? -(ra(rg) * v0 + rc(rg)) * ib : -rc(rg) * ib;
            w(LY::O_D, k) += 2.0 * qu * kc * ib;
            if (k >= 1) w(LY::O_D, k - 1) += 2.0 * qu * kc * ea;
            dual += qu * kc * kc;
        }
        double gr[N];
        HVP_FLAT_UNROLL
        for (int j = 0; j < N; ++j) gr[j] = w(LY::O_D, j);
        HVP_ROLL
        for (int i = 0; i < N; ++i) {
            double s = 0.0;
            HVP_FLAT_UNROLL
            for (int j = 0; j < N; ++j) s -= w(LY::O_HINV, i * N + j) * gr[j];
            if (ALG2) w(LY::O_R, i) = s - w(LY::O_X, i);    // x_u - x* (warm start: residuals of the parent's rows)
            w(LY::O_X, i) = s;
            dual += 0.5 * w(LY::O_D, i) * s;      // objective at the unconstrained minimiser: c + g'x/2
        }
        it = 0; satf = 0; satb = 0;
        state = S_SELECT;
#ifdef HVP_DEBUG_STATS
        g_warm[0] += 1; if (warm) g_warm[1] += 1;
#endif
        if (warm) {
            // residual c_a = n_a'x_u - rhs_a of the parent's rows: a bound row's right-hand side may have moved
            // (the region of the newly fixed stage), every other row was active at x*: c_a = n_a'(x_u - x*)
            SlotIter si = slots();
            HVP_ROLL
            for (int a = 0; a < q; ++a) {
                const int b = si.next(), j = b & 15;
                double cv;
                if ((b >> 5) == R_BOUND) {
                    double lo, hi;
                    bounds(j, lo, hi);
                    cv = (b & 16) ? lo - w(LY::O_X, j) : w(LY::O_X, j) - hi;     // LB : UB
                } else {
                    cv = slot_dot(b, LY::O_R);
                }
                w(LY::O_YP, a) = cv;
            }
            bool ok = true;
            double cl = 0.0;
            HVP_ROLL
            for (int a = 0; a < q; ++a) {                                    // lambda = Ginv c
                double s = 0.0;
                int gi = tri(a, 0);
                HVP_ROLL
                for (int b = 0; b <= a; ++b) s += w(LY::O_GINV, gi + b) * w(LY::O_YP, b);
                gi += 2 * a + 1;
                HVP_ROLL
                for (int b = a + 1; b < q; ++b) { s += w(LY::O_GINV, gi) * w(LY::O_YP, b); gi += b + 1; }
                w(LY::O_LAM, a) = s;
                cl += s * w(LY::O_YP, a);
                if (!(s >= 0.0) || (slot_soft(act_raw(a)) && s > ww)) ok = false;
            }
#ifdef HVP_DEBUG_STATS
            if (ok) g_warm[2] += 1; was_warm = ok;
#endif
            if (ok) {
                // x = x_u - H^-1 N lambda ; dual value = f(x_u) + c'lambda / 2
                HVP_ROLL
                for (int i = 0; i < N; ++i) w(LY::O_WV, i) = 0.0;
                SlotIter sj = slots();
                HVP_ROLL
                for (int a = 0; a < q; ++a) slot_axpy(sj.next(), w(LY::O_LAM, a), LY::O_WV);
                double wr[N];
                HVP_FLAT_UNROLL
                for (int j = 0; j < N; ++j) wr[j] = w(LY::O_WV, j);
                HVP_ROLL
                for (int i = 0; i < N; ++i) {
                    double s = 0.0;
                    HVP_FLAT_UNROLL
                    for (int j = 0; j < N; ++j) s += w(LY::O_HINV, i * N + j) * wr[j];
                    w(LY::O_X, i) -= s;
                }
                dual += 0.5 * cl;
                it = 1;
                if (dual > inc) node_done(1, 0.0);                          // dual-bound pruning, as in do_step
                return;
            }
        }
        q = 0; act_lo = act_hi = 0;
    }

    // merged simple bounds of x_j = v_{j+1}: state box, region of stage j+1 if fixed, stage-0 rows
    HVP_HD void bounds(int j, double& lo, double& hi) const {
        lo = P->vmin; hi = P->vmax;
        if (kHull && j >= L) { lo = fmax(lo, C->rlo[j + 1]); hi = fmin(hi, C->rhi[j + 1]); }
        if (j + 1 < L) {
            const int rg = mode(j + 1);
            lo = nmax(lo, P->edge[rg]); hi = nmin(hi, P->edge[rg + 1]);
        }
        if (j == 0) {
            const int r0 = mode(0);
            const double m = ra(r0) * v0 + rc(r0), bb = rb(r0);
            lo = nmax(lo, nmax(v0 + P->a_dec, m + bb * P->umin));
            hi = nmin(hi, nmin(v0 + P->a_acc, m + bb * P->umax));
        }
    }

    // ---- SELECT: most violated row, or the node is solved ---------------------------------
    HVP_HD void do_select() {
        const double tol = 1e-9;
        const double qu = P->qu, ww = P->w;
        double best = tol; int bid = -1;
        double PS = 0.0, xm = v0;
        // The scan is UNROLLED over the stages and every stage keeps its own (best, id) pair: a rolled loop is one
        // serial chain of ~8 N compare-selects (r01k ncu: a third of all stall samples sit on this scan, almost
        // all fixed-latency dependency waits); unrolled, the N stage chains are independent and interleave, stage
        // indices become immediates, and the soft-row loads are all issued up front.  The combination below keeps
        // the first row that attains the maximum, exactly as the single chain did.
        double bj[N]; int ij[N];
#define HVP_CAND(T, J, S)                                              \
    {                                                                  \
        const double s__ = (S);                                        \
        if (s__ > lb) { lb = s__; li = (T) * 16 + (J); }               \
    }
        HVP_FLAT_UNROLL
        for (int j = 0; j < N; ++j) {
            double lb = tol; int li = -1;
            const double xv = w(LY::O_X, j);
            double lo, hi;
            bounds(j, lo, hi);
            HVP_CAND(T_UB, j, xv - hi);
            HVP_CAND(T_LB, j, lo - xv);
            if (j >= 1) {
                if (j < L) {
                    const int rg = mode(j);
                    const double du = xv - ra(rg) * xm - rc(rg), bb = rb(rg);
                    HVP_CAND(T_UHI, j, du - bb * P->umax);
                    HVP_CAND(T_ULO, j, bb * P->umin - du);
                }
                const double dv = xv - xm;
                HVP_CAND(T_ACC, j, dv - ((j < L || !kHull) ? P->a_acc - j * P->tight : C->amax[j]));
                HVP_CAND(T_DEC, j, ((j < L || !kHull) ? P->a_dec + j * P->tight : C->amin[j]) - dv);
                if (has_sf) {
                    const double s = PS - sfv[j];
                    HVP_CAND(T_SF, j, ((satf >> j) & 1u) ? -s : s);
                }
                if (has_sb) {
                    const double s = sbv[j] - PS;
                    HVP_CAND(T_SB, j, ((satb >> j) & 1u) ? -s : s);
                }
                // position box: prefix sums increase with j once the velocity bounds hold, so the
                // smallest (j = 1) and largest (j = N-1) are the rows that can stay violated
                if (j == 1) HVP_CAND(T_PLO, j, (P->pmin - pc) - PS);
                if (j == N - 1) HVP_CAND(T_PHI, j, PS - (P->pmax - pc));
            }
            PS += xv; xm = xv;
            bj[j] = lb; ij[j] = li;
        }
        HVP_FLAT_UNROLL
        for (int j = 0; j < N; ++j)
            if (bj[j] > best) { best = bj[j]; bid = ij[j]; }
#undef HVP_CAND
        if (bid >= 0) {
            // p = row (type pt, stage pj) and the slot byte it will have (act_raw)
            const int pt = bid >> 4;
            pj = bid & 15;
            int cls = (int)((kClassOfType >> (4 * pt)) & 7u);
            if (cls == R_IN_LO && mode(pj) >= 4) cls = R_IN_HI;
            pkind = cls == R_BOUND ? 0 : (cls < R_POS ? 1 : 2);
            psgn = (pt & 1) ? -1.0 : 1.0;
            if (pt == T_SF) psgn = ((satf >> pj) & 1u) ? -1.0 : 1.0;
            if (pt == T_SB) psgn = ((satb >> pj) & 1u) ? 1.0 : -1.0;
            pcode = pj | (psgn < 0.0 ? 16 : 0) | (cls << 5);
            pcoef = slot_coef(pcode);
            p_soft = cls >= R_SF;
            // The most violated row is already active: its residual is round-off drift (ill-conditioned,
            // heavily constrained node) and every other row is violated by even less -> converged.
            bool dup = false;
            SlotIter si = slots();
            HVP_ROLL
            for (int a = 0; a < q; ++a) dup = dup || (si.next() == pcode);
            if (dup) {
                if (best < 1e-6) bid = -1;
                else { node_done(2, 0.0); return; }
            }
        }
        if (bid < 0) {
            // ---- node solved: objective = tracking closed form + input cost + L1 penalties ----
            double f = ct;
            PS = 0.0; xm = v0;
            HVP_FLAT_UNROLL
            for (int j = 0; j < N; ++j) {
                const double xv = w(LY::O_X, j);
                f += xv * (0.5 * Hdiag(j) * xv + Hoff(j) * PS + C->gt[j]);
                if (j < L) {
                    const int rg = mode(j);
                    const double uu = (xv - ra(rg) * xm - rc(rg)) * hvp_rcp(rb(rg));
                    f += qu * uu * uu;
                }
                if (j >= 1) {
                    if (has_sf) { const double s = PS - sfv[j]; if (s > 0) f += ww * s; }
                    if (has_sb) { const double s = sbv[j] - PS; if (s > 0) f += ww * s; }
                }
                PS += xv; xm = xv;
            }
            node_done(0, f);
            return;
        }
        // yp = H^-1 n_p and nHn = n_p' yp
        double acc = 0.0;
        HVP_ROLL
        for (int i = 0; i < N; ++i) {
            double s;
            if (pkind == 0) s = w(LY::O_HINV, pj * N + i);
            else if (pkind == 1) s = w(LY::O_HINV, pj * N + i) - pcoef * w(LY::O_HINV, (pj - 1) * N + i);
            else {
                s = 0.0;
                HVP_ROLL
                for (int k = 0; k < pj; ++k) s += w(LY::O_HINV, k * N + i);
            }
            s *= psgn;
            w(LY::O_YP, i) = s;
            // n_p' yp accumulates with the same structure
            if (pkind == 0) acc += (i == pj) ? s : 0.0;
            else if (pkind == 1) acc += (i == pj) ? s : ((i == pj - 1) ? -pcoef * s : 0.0);
            else acc += (i < pj) ? s : 0.0;
        }
        nHn = psgn * acc;
        cp = best;
        lam_p = 0.0;
        state = S_STEP;
    }

    // n' v for the row of slot byte b, v in the work array at `off`
    HVP_HD double slot_dot(int b, int off) const {
        const int j = b & 15, cls = b >> 5;
        double s;
        if (cls == R_BOUND) s = w(off, j);
        else if (cls < R_POS) s = w(off, j) - slot_coef(b) * w(off, j - 1);
        else {
            s = 0.0;
            HVP_ROLL
            for (int i = 0; i < j; ++i) s += w(off, i);
        }
        return (b & 16) ? -s : s;
    }
    HVP_HD void slot_axpy(int b, double c0, int off) const {
        const int j = b & 15, cls = b >> 5;
        const double c = (b & 16) ? -c0 : c0;
        if (cls == R_BOUND) w(off, j) += c;
        else if (cls < R_POS) { w(off, j) += c; w(off, j - 1) -= c * slot_coef(b); }
        else {
            HVP_ROLL
            for (int i = 0; i < j; ++i) w(off, i) += c;
        }
    }

    // ---- STEP: one primal-dual step towards adding p ----------------------------------------
    HVP_HD void do_step() {
        const double tol = 1e-9, ww = P->w;
        if (++it > 40 * N + 60) { node_done(2, 0.0); return; }
        // p can reach its boundary exactly at the end of a PARTIAL step (t1 = t2 tie): it then joins the
        // active set with the multiplier it has accumulated (a full step of length zero) -- returning to
        // SELECT here would drop lam_p * n_p from the stationarity condition
        const bool zero_step = (cp <= tol);
        if (zero_step && !(lam_p > 0.0)) { state = S_SELECT; return; }
        // d = N' yp ; r = Ginv d ; nz = nHn - d'r
        SlotIter si = slots();
        HVP_ROLL
        for (int a = 0; a < q; ++a) w(LY::O_D, a) = slot_dot(si.next(), LY::O_YP);
        double nz = nHn;
        // ratio tests without a division per slot: keep the best (numerator, denominator) pair
        double n1 = 1.0, d1 = 0.0, n3 = 1.0, d3 = 0.0;
        int k1 = -1, k3 = -1;
        HVP_ROLL
        for (int a = 0; a < q; ++a) {
            double s = 0.0;
            int gi = tri(a, 0);                            // row a of the packed symmetric matrix: b <= a contiguous ...
            HVP_ROLL
            for (int b = 0; b <= a; ++b) s += w(LY::O_GINV, gi + b) * w(LY::O_D, b);
            gi += 2 * a + 1;                               // ... then down column a: tri(b, a), stride b + 1
            HVP_ROLL
            for (int b = a + 1; b < q; ++b) { s += w(LY::O_GINV, gi) * w(LY::O_D, b); gi += b + 1; }
            w(LY::O_R, a) = s;
            nz -= s * w(LY::O_D, a);
            const double la = w(LY::O_LAM, a);
            if (s > 1e-14) {
                if (k1 < 0 || la * d1 < n1 * s) { n1 = la; d1 = s; k1 = a; }
            } else if (s < -1e-14 && slot_soft(act_raw(a))) {
                const double num = ww - la, den = -s;
                if (k3 < 0 || num * d3 < n3 * den) { n3 = num; d3 = den; k3 = a; }
            }
        }
        const bool dependent = (q == N) || !(nz > 1e-11 * nHn);
        const double INF = HUGE_VAL;
        if (zero_step && dependent) { node_done(2, 0.0); return; }
        const double t2 = dependent ? INF : (zero_step ? 0.0 : cp * hvp_rcp(nz));
        const double t1 = k1 >= 0 ? n1 * hvp_rcp(d1) : INF;
        const double t3 = k3 >= 0 ? n3 * hvp_rcp(d3) : INF;
        const double t3p = p_soft ? (ww - lam_p) : INF;
        const double t = fmin(fmin(t1, t2), fmin(t3, t3p));
        if (!(t < INF)) { node_done(1, 0.0); return; }          // infeasible node
        // the dual value grows by the violation of p integrated along the step; it bounds the node
        // optimum from below, so a node whose dual passes the incumbent is finished
        dual += t * cp - (dependent ? 0.0 : 0.5 * t * t * nz);
        if (dual > inc) { node_done(1, 0.0); return; }
        if (!dependent) {
            // w = n_p - N r ;  x -= t H^-1 w ;  the violation of p shrinks by t * nz
            HVP_ROLL
            for (int i = 0; i < N; ++i) {
                double v;
                if (pkind == 0) v = (i == pj) ? psgn : 0.0;
                else if (pkind == 1) v = (i == pj) ? psgn : ((i == pj - 1) ? -psgn * pcoef : 0.0);
                else v = (i < pj) ? psgn : 0.0;
                w(LY::O_WV, i) = v;
            }
            SlotIter sj = slots();
            HVP_ROLL
            for (int a = 0; a < q; ++a) slot_axpy(sj.next(), -w(LY::O_R, a), LY::O_WV);
            double wr[N];
            HVP_FLAT_UNROLL
            for (int j = 0; j < N; ++j) wr[j] = w(LY::O_WV, j);
            HVP_ROLL
            for (int i = 0; i < N; ++i) {
                double s = 0.0;
                HVP_FLAT_UNROLL
                for (int j = 0; j < N; ++j) s += w(LY::O_HINV, i * N + j) * wr[j];
                w(LY::O_X, i) -= t * s;
            }
            cp -= t * nz;
        }
        HVP_ROLL
        for (int a = 0; a < q; ++a) w(LY::O_LAM, a) -= t * w(LY::O_R, a);
        lam_p += t;
        if (t == t2) {
            // p becomes slot q: bordering update of Ginv with Schur complement nz
            const double is = hvp_rcp(nz);
            HVP_ROLL
            for (int a = 0; a < q; ++a) {
                const double ra_ = w(LY::O_R, a) * is;
                HVP_ROLL
                for (int b = 0; b <= a; ++b) w(LY::O_GINV, tri(a, b)) += ra_ * w(LY::O_R, b);
                w(LY::O_GINV, tri(q, a)) = -ra_;
            }
            w(LY::O_GINV, tri(q, q)) = is;
            set_act(q, pcode);
            w(LY::O_LAM, q) = lam_p;
            ++q;
            state = S_SELECT;
            return;
        }
        if (t == t3p) {                                          // soft p saturates: flip, not added
            if ((pcode >> 5) == R_SF) satf ^= (1u << pj); else satb ^= (1u << pj);
            state = S_SELECT;
            return;
        }
        int drop;
        if (t == t1) drop = k1;
        else {                                                   // active soft row saturates: flip + drop
            drop = k3;
            const int b = act_raw(drop), j = b & 15;
            if ((b >> 5) == R_SF) satf ^= (1u << j); else satb ^= (1u << j);
        }
        {   // Ginv <- Ginv - g_k g_k'/g_kk, then delete row/column `drop` (packed, in place)
            const double ikk = hvp_rcp(w(LY::O_GINV, tri(drop, drop)));
            HVP_ROLL
            for (int a = 0; a < q; ++a) w(LY::O_D, a) = w(LY::O_GINV, a >= drop ? tri(a, drop) : tri(drop, a));
            HVP_ROLL
            for (int a = 0; a < q; ++a) {
                if (a == drop) continue;
                const int an = a > drop ? a - 1 : a;
                const double da = w(LY::O_D, a) * ikk;
                HVP_ROLL
                for (int b = 0; b <= a; ++b) {
                    if (b == drop) continue;
                    const int bn = b > drop ? b - 1 : b;
                    w(LY::O_GINV, tri(an, bn)) = w(LY::O_GINV, tri(a, b)) - da * w(LY::O_D, b);
                }
            }
        }
        HVP_ROLL
        for (int a = drop; a + 1 < q; ++a) {
            set_act(a, act_raw(a + 1));
            w(LY::O_LAM, a) = w(LY::O_LAM, a + 1);
        }
        --q;
        // state stays S_STEP: continue with the same p
    }

    HVP_HD void trip() {
        if (state == S_NEXT) do_next();
        if (state == S_BUILD) do_build();
        if (state == S_SELECT) do_select();
        if (state == S_STEP) do_step();
    }
    // the two halves of a trip, so that a warp can run the (expensive, once per node) node set-up for
    // MANY lanes at once instead of for the one or two lanes that happen to need it on every trip
    HVP_HD bool wants_node() const { return state == S_NEXT || state == S_BUILD; }
    HVP_HD void trip_node() {
        if (state == S_NEXT) do_next();
        if (state == S_BUILD) do_build();
    }
    HVP_HD void trip_step() {
        if (state == S_SELECT) do_select();
        if (state == S_STEP) do_step();
    }

    // ---- results: best_ (= x_out + N + 2) already holds the incumbent velocities v_1..v_N -------
    HVP_HD LocalResult finish(double* u_out, double* x_out, int32_t* mode_out) const {
        LocalResult R;
        R.nodes = nodes; R.qp_iters = iters;
        const int np1 = N + 1;
        if (inc < HUGE_VAL) {
            R.obj = inc;
            R.status = timeout ? HVP_ST_TIME_LIMIT : limit ? HVP_ST_NODE_LIMIT : (trouble ? HVP_ST_NUMERIC : HVP_ST_OPTIMAL);
            double p = p0, v = v0;
            x_out[0] = p; x_out[np1] = v;
            HVP_ROLL
            for (int k = 0; k < N; ++k) {
                const int rg = mode_of(best_modes, k);
                const double vn = x_out[np1 + k + 1];
                u_out[k] = (vn - ra(rg) * v - rc(rg)) / rb(rg);
                mode_out[k] = rg;
                p = p + v; v = vn;
                x_out[k + 1] = p;
            }
        } else {
            R.obj = HUGE_VAL;
            R.status = timeout ? HVP_ST_TIME_LIMIT : limit ? HVP_ST_NODE_LIMIT : (trouble ? HVP_ST_NUMERIC : HVP_ST_INFEASIBLE);
            HVP_ROLL
            for (int k = 0; k < N; ++k) { u_out[k] = 0.0; mode_out[k] = -1; }
            HVP_ROLL
            for (int k = 0; k <= N; ++k) { x_out[k] = 0.0; x_out[np1 + k] = 0.0; }
        }
        return R;
    }
};

}  // namespace hvp
