// coop_core.cuh -- per-vehicle local hybrid-MPC MIQP solved COOPERATIVELY by a group of G lanes.
//
// Same mathematics as miqp_core.cuh (velocity-space node QPs, bounded-dual Goldfarb-Idnani with
// exact L1 slack elimination, depth-first branch-and-bound with relaxed-tail bounds; problem
// definition fleet_decent_mld.py:61-208 on the pwa_gear model, models.py:397-492), re-laid-out
// for the warp:
//   * lane j of the group owns velocity variable x_j, row j of H^-1, row j of Y = H^-1 N and, as
//     "slot" j of the active set, row j of (N'H^-1N)^-1 with that constraint's multiplier --
//     everything in registers, no shared or local memory;
//   * matrix-vector products are G FMAs per lane, reductions / broadcasts / prefix sums are warp
//     shuffles restricted to the group; the violation scan is parallel over the horizon;
//   * every branch is taken on group-uniform values, so a group never diverges internally; with
//     G = 8 a warp carries four independent problems.
// Written against the backend vocabulary of coop_backend.cuh (DevBK on the GPU; HostBK emulates
// the same lane program on the CPU for the tests).
#pragma once
#include "coop_backend.cuh"
#include "miqp_core.cuh"   // LocalParams, LocalResult, status codes, constraint type ids

#if defined(__CUDACC__)
#define HVP_CD __device__ __forceinline__
#else
#define HVP_CD inline
#endif

namespace hvp {

template <class BK>
struct CoopSolver {
    static constexpr int G = BK::G;
    using D = typename BK::D;
    using I = typename BK::I;
    using Bm = typename BK::Bm;

    BK bk;
    const LocalParams* P;
    int N, flags;
    double p0, v0, pc;
    double inv_m, a_lo, a_hi, c_lo, c_hi;
    double hw1, hw2, hd, ct;
    bool has_sf, has_sb;
    // distributed over lanes: element j on lane j
    D x, gt, lb, ub, sf, sb, best;
    D xstar;            // level lev on lane lev (lev = 0..N-1)
    D rlo, rhi;         // level lev (1..N) on lane lev-1; level 0 is [v0, v0]
    D hinv[G];          // row j of H^-1
    D Y[G];             // row j of Y = H^-1 N   (column a = active slot a)
    D ginv[G];          // slot a on lane a: row a of (N'H^-1N)^-1
    D lam, s_sgn, s_coef;
    I s_kind, s_j, s_id;
    // group-uniform
    int L, q, iters;
    uint64_t modes_pk, am_lo, am_hi;
    uint32_t satf, satb;

    HVP_CD double ra(int rg) const { return rg < 4 ? a_lo : a_hi; }
    HVP_CD double rc(int rg) const { return rg < 4 ? c_lo : c_hi; }
    HVP_CD double rb(int rg) const { return P->bgear[rg] * inv_m; }
    HVP_CD int mode(int k) const { return (int)((modes_pk >> (3 * k)) & 7u); }
    HVP_CD void set_mode(int k, int rg) { modes_pk = (modes_pk & ~(7ull << (3 * k))) | ((uint64_t)rg << (3 * k)); }
    HVP_CD void mark(int id, bool on) {
        if (id < 64) am_lo = on ? (am_lo | (1ull << id)) : (am_lo & ~(1ull << id));
        else am_hi = on ? (am_hi | (1ull << (id - 64))) : (am_hi & ~(1ull << (id - 64)));
    }
    // per-lane versions of the region data for per-lane region index rg
    HVP_CD D ra_l(const I& rg) const { return bk.sel(rg < 4, bk.splat(a_lo), bk.splat(a_hi)); }
    HVP_CD D rc_l(const I& rg) const { return bk.sel(rg < 4, bk.splat(c_lo), bk.splat(c_hi)); }
    HVP_CD D rb_l(const I& rg) const { return bk.lookup(P->bgear, rg) * inv_m; }

    // -------------------------------------------------------------------------------------
    HVP_CD void setup(const LocalParams* P_, int flags_, double mass, const double* x0, const double* xf,
                      const double* xb, const double* xl) {
        P = P_; N = P->N; flags = flags_;
        p0 = x0[0]; v0 = x0[1]; pc = p0 + v0;
        inv_m = 1.0 / mass;
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
        // no reference term (a front vehicle that is also the trailer and not the leader): the Hessian is the input
        // cost of the fixed stages alone, singular at every node that leaves a stage free -- only leaves are solved
        notrack = nterm < 0.5;
        const I ln = bk.lane();
        const Bm valid = ln < N;
        const I kk = ln + 1;                       // lane j holds stage k = j+1
        gt = bk.splat(0.0);
        ct = 0.0;
        for (int kind = 0; kind < 3; ++kind) {
            const double* ref = kind == 0 ? xf : (kind == 1 ? xb : xl);
            const bool on = kind == 0 ? tf : (kind == 1 ? tb : tl);
            if (!on) continue;
            const double tau = kind == 0 ? t0 : 0.0;
            const D pk = bk.ld(ref, kk, valid), vk = bk.ld(ref, kk + np1, valid);
            const D Pk = (kind == 0) ? (pk - d0) : (kind == 1) ? (pk + t0 * vk + d0) : pk;
            const D rho = bk.sel(valid, pc - Pk, bk.splat(0.0));
            const double total = bk.gsum(rho);
            const D suffix = total - (bk.scan_excl(rho) + rho);       // sum over later stages
            gt += bk.sel(valid, 2.0 * wp * (suffix + tau * rho) - 2.0 * wvv * vk, bk.splat(0.0));
            ct += bk.gsum(bk.sel(valid, wp * rho * rho + wvv * vk * vk, bk.splat(0.0)));
            const double pk0 = ref[0], vk0 = ref[np1];
            const double Pk0 = (kind == 0) ? (pk0 - d0) : (kind == 1) ? (pk0 + t0 * vk0 + d0) : pk0;
            const double e0 = p0 + tau * v0 - Pk0, e1 = v0 - vk0;
            ct += wp * e0 * e0 + wvv * e1 * e1;
        }
        has_sf = !is_front; has_sb = !is_trailer;
        const double ww = P->w, ds = P->d_safe;
        sf = bk.splat(0.0); sb = bk.splat(0.0);
        const Bm srow = (ln >= 1) & valid;          // rows j = 1..N-1 use stage k = j+1
        if (has_sf) {
            const double s0 = p0 - (xf[0] - ds), s1 = pc - (xf[1] - ds);
            ct += ww * (s0 > 0 ? s0 : 0.0) + ww * (s1 > 0 ? s1 : 0.0);
            sf = bk.ld(xf, kk, srow) - ds - pc;
        }
        if (has_sb) {
            const double s0 = (xb[0] + ds) - p0, s1 = (xb[1] + ds) - pc;
            ct += ww * (s0 > 0 ? s0 : 0.0) + ww * (s1 > 0 ? s1 : 0.0);
            sb = bk.ld(xb, kk, srow) + ds - pc;
        }
    }

    // coefficient of structured row (kind, j, sgn, coef) at column c  (group-uniform)
    HVP_CD static double coef_at(int kind, int j, double sgn, double coef, int c) {
        if (kind == 0) return c == j ? sgn : 0.0;
        if (kind == 1) return c == j ? sgn : (c == j - 1 ? -sgn * coef : 0.0);
        return c < j ? sgn : 0.0;
    }

    // =====================================================================================
    // Flat state machine.  One trip of the loop in run() executes, in this order and each at most
    // once: NEXT (branch-and-bound bookkeeping) -> BUILD (node Hessian, H^-1, unconstrained
    // minimiser) -> SELECT (violation scan / node finished) -> STEP (one dual active-set step).
    // The four groups of a warp all run this same loop, so whatever their individual progress they
    // re-converge at every block boundary instead of serialising whole solves.
    // =====================================================================================
    enum : int { S_NEXT = 0, S_BUILD, S_SELECT, S_STEP, S_DONE };

    // persistent across trips -------------------------------------------------------------
    int state, lev, it, nodes;
    double inc, nlo_cur, nhi_cur;
    double dual;                 // value of the node's dual function: lower bound on the node optimum
    bool dive;                   // first descent: path nodes are not solved, only the leaf
    bool notrack;                // no reference term: no node but a leaf is solved (setup)
    uint64_t best_modes, cand_lo, cand_hi;
    bool trouble, limit, timeout;
    long long t_start;
    // ---- one tree searched by several workers (latency path: a scenario-timestep is ten MIQPs, the GPU has room for a
    // hundred warps).  Every worker runs the SAME root relaxation and first dive -- deterministic, so all of them hold
    // the same depth-first stack and the same first incumbent -- and from there the sub-trees that hang off the dive
    // path are dealt round robin: the k-th sibling popped ON the path belongs to worker k mod sub_M, whoever owns it
    // searches it completely.  path_lev = deepest level still on the path (a pop at a deeper level is inside an owned
    // sub-tree).  The workers share their incumbent through `shared` (atomicMin on an order-preserving key).
    int sub_M = 1, sub_w = 0, sub_cnt = 0, path_lev = 1 << 20;
    double own = HUGE_VAL;                  // objective of THIS worker's best leaf (inc may be another worker's)
    unsigned long long* shared = nullptr;
    // constraint being added
    int pid, pkind, pj;
    double psgn, pcoef, prhs, nHn, lam_p;
    bool p_soft;
    D np, yp, yps;

    HVP_CD static int cand_get(uint64_t lo, uint64_t hi, int lv) {
        const unsigned sh = (unsigned)(7 * (lv < 9 ? lv : lv - 9));
        return (int)(((lv < 9 ? lo : hi) >> sh) & 0x7fu);
    }
    HVP_CD static void cand_set(uint64_t& lo, uint64_t& hi, int lv, int val) {
        const unsigned sh = (unsigned)(7 * (lv < 9 ? lv : lv - 9));
        uint64_t& t = lv < 9 ? lo : hi;
        t = (t & ~(0x7full << sh)) | ((uint64_t)val << sh);
    }

    HVP_CD void begin() {
        iters = 0; modes_pk = 0; nodes = 0; it = 0;
        inc = HUGE_VAL; best_modes = 0; cand_lo = cand_hi = 0; trouble = limit = timeout = false; dive = P->dive != 0; t_start = P->time_limit_ns > 0 ? hvp_now_ns() : 0;
        best = bk.splat(0.0); xstar = bk.splat(v0); rlo = bk.splat(0.0); rhi = bk.splat(0.0);
        lev = 0;
        int c0 = 0;
        for (int rg = 0; rg < NREG; ++rg)
            if (v0 >= P->edge[rg] && v0 <= P->edge[rg + 1]) c0 |= (1 << rg);
        cand_set(cand_lo, cand_hi, 0, c0);
        state = S_NEXT;
        sub_cnt = 0; own = HUGE_VAL;
        path_lev = dive ? (1 << 20) : 0;             // no dive: the path is the root, its candidates are dealt at once
    }

    // ---- NEXT: pick the next node of the depth-first search (or finish) -------------------
    HVP_CD void do_next() {
        const double eps = 1e-9;
        const I ln = bk.lane();
        for (;;) {
            int cset = cand_get(cand_lo, cand_hi, lev);
            if (cset == 0) {
                if (lev == 0) { state = S_DONE; return; }
                --lev;
                continue;
            }
            int rg = -1; double bd = HUGE_VAL;
            const double xs = bk.bcast(xstar, lev);
            for (int c = 0; c < NREG; ++c) {
                if (!((cset >> c) & 1)) continue;
                const double lo = P->edge[c], hi = P->edge[c + 1];
                const double dist = xs < lo ? lo - xs : (xs > hi ? xs - hi : 0.0);
                if (dist < bd) { bd = dist; rg = c; }
            }
            cset &= ~(1 << rg);
            cand_set(cand_lo, cand_hi, lev, cset);
            if (sub_M > 1 && !dive) {
                if (lev < path_lev) path_lev = lev;
                if (lev == path_lev && (sub_cnt++ % sub_M) != sub_w) continue;      // another worker's sub-tree
            }
            set_mode(lev, rg);
            const double cur_lo = lev == 0 ? v0 : bk.bcast(rlo, lev - 1);
            const double cur_hi = lev == 0 ? v0 : bk.bcast(rhi, lev - 1);
            const double jlo = fmax(cur_lo, P->edge[rg]), jhi = fmin(cur_hi, P->edge[rg + 1]);
            if (jlo > jhi + eps) continue;
            double nlo = fmax(ra(rg) * jlo + rc(rg) + rb(rg) * P->umin, jlo + P->a_dec + lev * P->tight);
            double nhi = fmin(ra(rg) * jhi + rc(rg) + rb(rg) * P->umax, jhi + P->a_acc - lev * P->tight);
            nlo = fmax(nlo, P->vmin); nhi = fmin(nhi, P->vmax);
            if (nlo > nhi + eps) continue;
            if (pc > P->pmax + eps || pc < P->pmin - eps) continue;
            nlo_cur = nlo; nhi_cur = nhi;
            rlo = bk.sel(ln == lev, bk.splat(nlo - eps), rlo);
            rhi = bk.sel(ln == lev, bk.splat(nhi + eps), rhi);
            L = lev + 1;
            if (((dive && nodes >= 1) || notrack) && L < N) {
                // first descent (see flat_core.cuh): without an incumbent the relaxations along the path
                // cannot prune; follow the last relaxed trajectory and solve the leaf directly
                ++lev;
                xstar = bk.sel(ln == lev, bk.splat(notrack ? bk.bcast(xstar, lev - 1) : bk.bcast(x, lev - 1)), xstar);
                int cn = 0;
                for (int c = 0; c < NREG; ++c)
                    if (P->edge[c] <= nhi_cur + eps && P->edge[c + 1] >= nlo_cur - eps) cn |= (1 << c);
                cand_set(cand_lo, cand_hi, lev, cn);
                continue;
            }
            // merged simple bounds: state box, regions of fixed stages, stage-0 accel/input rows
            const I rgn = bk.bits3(modes_pk, ln + 1);
            const Bm fixed = (ln + 1) < L;
            const D elo = bk.lookup(P->edge, rgn), ehi = bk.lookup(P->edge, rgn + 1);
            lb = bk.sel(fixed, bk.dmax(bk.splat(P->vmin), elo), bk.splat(P->vmin));
            ub = bk.sel(fixed, bk.dmin(bk.splat(P->vmax), ehi), bk.splat(P->vmax));
            const int r0 = mode(0);
            const double l0 = fmax(v0 + P->a_dec, ra(r0) * v0 + rc(r0) + rb(r0) * P->umin);
            const double u0 = fmin(v0 + P->a_acc, ra(r0) * v0 + rc(r0) + rb(r0) * P->umax);
            lb = bk.sel(ln == 0, bk.dmax(lb, bk.splat(l0)), lb);
            ub = bk.sel(ln == 0, bk.dmin(ub, bk.splat(u0)), ub);
            state = S_BUILD;
            return;
        }
    }

    // incumbent exchange between the workers of one tree (device only; a single worker / the host build: no-ops)
    HVP_CD void share_in() {
#if defined(__CUDA_ARCH__)
        if (shared) {
            const unsigned long long k = *reinterpret_cast<volatile unsigned long long*>(shared);
            const double g = hvp_key2d(k);
            if (g < inc) inc = g;
        }
#endif
    }
    HVP_CD void share_out() {
#if defined(__CUDA_ARCH__)
        if (shared) atomicMin(shared, hvp_d2key(own));
#endif
    }

    // outcome of a node: st 0 solved (obj valid), 1 infeasible, 2 numeric trouble
    HVP_CD void node_done(int st, double obj) {
        iters += it;
        ++nodes;
        state = S_NEXT;
        if (dive && (st != 0 || L == N)) { dive = false; path_lev = lev; }           // the dive ends here: the path is known
        if (st != 0 || L == N) dive = false;
        if (st == 2) { trouble = true; return; }
        if (st == 1) return;
        share_in();
        if (inc < HUGE_VAL && !(obj < hvp_cut(inc, P->mip_gap))) return;              // bound
        if (L == N) { inc = obj; own = obj; best = x; best_modes = modes_pk; share_out(); return; }   // leaf
        if (P->max_nodes > 0 && nodes >= P->max_nodes) { limit = true; state = S_DONE; return; }
        if (P->time_limit_ns > 0 && hvp_now_ns() - t_start > P->time_limit_ns) { timeout = true; state = S_DONE; return; }
        const double eps = 1e-9;
        const I ln = bk.lane();
        ++lev;
        xstar = bk.sel(ln == lev, bk.splat(bk.bcast(x, lev - 1)), xstar);
        int cn = 0;
        for (int c = 0; c < NREG; ++c)
            if (P->edge[c] <= nhi_cur + eps && P->edge[c + 1] >= nlo_cur - eps) cn |= (1 << c);
        cand_set(cand_lo, cand_hi, lev, cn);
    }

    // ---- BUILD: Hessian rows, in-place Gauss-Jordan inverse, unconstrained minimiser -------
    HVP_CD void do_build() {
        const double qu = P->qu;
        const I ln = bk.lane();
        const Bm valid = ln < N;
        const D lnd = bk.todouble(ln);
        const D hoff_l = hw1 * ((double)(N - 1) - lnd) + hw2;     // H_t[i][j], i<j, depends on j only
        const D hdiag_l = hw1 * ((double)(N - 1) - lnd) + hd;
        D g = gt;
        double kc2 = 0.0;
#pragma unroll
        for (int c = 0; c < G; ++c) {
            const double hoff_c = hw1 * (double)(N - 1 - c) + hw2;
            D h = bk.sel(ln > c, hoff_l, bk.splat(hoff_c));
            h = bk.sel(ln == c, hdiag_l, h);
            h = bk.sel(valid & (c < N), h, bk.sel(ln == c, bk.splat(1.0), bk.splat(0.0)));   // padding: identity
            hinv[c] = h;
        }
        // input cost of fixed stages: u_k = (x_k - a x_{k-1} - c)/b   (x_{-1} = v0)
#pragma unroll
        for (int k = 0; k < G; ++k) {
            if (k < L) {
                const int rg = mode(k);
                const double ib = bk.sdiv(1.0, rb(rg)), ea = -ra(rg) * ib;
                const double kc = (k == 0) ? -(ra(rg) * v0 + rc(rg)) * ib : -rc(rg) * ib;
                hinv[k] += bk.sel(ln == k, bk.splat(2.0 * qu * ib * ib), bk.splat(0.0));
                g += bk.sel(ln == k, bk.splat(2.0 * qu * kc * ib), bk.splat(0.0));
                kc2 += qu * kc * kc;
                if (k >= 1) {
                    hinv[k] += bk.sel(ln == k - 1, bk.splat(2.0 * qu * ea * ib), bk.splat(0.0));
                    hinv[k - 1] += bk.sel(ln == k, bk.splat(2.0 * qu * ea * ib),
                                          bk.sel(ln == k - 1, bk.splat(2.0 * qu * ea * ea), bk.splat(0.0)));
                    g += bk.sel(ln == k - 1, bk.splat(2.0 * qu * kc * ea), bk.splat(0.0));
                }
            }
        }
        bool bad = false;
#pragma unroll
        for (int k = 0; k < G; ++k) {
            if (k < N) {
                const double piv = bk.bcast(hinv[k], k);
                bad = bad || !(piv > 0.0);
                const double pinv = bk.sdiv(1.0, piv);
                const D f = hinv[k];
                const Bm isk = ln == k;
#pragma unroll
                for (int c = 0; c < G; ++c) {
                    if (c == k) continue;
                    const double rk = bk.bcast(hinv[c], k) * pinv;
                    hinv[c] = bk.sel(isk, bk.splat(rk), hinv[c] - f * rk);
                }
                hinv[k] = bk.sel(isk, bk.splat(pinv), -(f * pinv));
            }
        }
        it = 0;
        if (bad) { node_done(2, 0.0); return; }
        D acc = bk.splat(0.0);
#pragma unroll
        for (int c = 0; c < G; ++c) acc -= hinv[c] * bk.bcast(g, c);
        x = bk.sel(valid, acc, bk.splat(0.0));
        dual = ct + kc2 + 0.5 * bk.gsum(bk.sel(valid, g * x, bk.splat(0.0)));   // objective at the unconstrained minimiser
        q = 0; satf = 0; satb = 0; am_lo = am_hi = 0;
        lam = bk.splat(0.0); s_sgn = bk.splat(0.0); s_coef = bk.splat(0.0);
        s_kind = bk.splati(0); s_j = bk.splati(0); s_id = bk.splati(0);
#pragma unroll
        for (int c = 0; c < G; ++c) { Y[c] = bk.splat(0.0); ginv[c] = bk.splat(0.0); }
        state = S_SELECT;
    }

    // ---- SELECT: most violated row, or the node is solved ---------------------------------
    HVP_CD void do_select() {
        const double tol = 1e-9;
        const double qu = P->qu, ww = P->w;
        const I ln = bk.lane();
        const Bm valid = ln < N;
        const D lnd = bk.todouble(ln);
        const D accmax = P->a_acc - lnd * P->tight, decmin = P->a_dec + lnd * P->tight;
        const D NEG = bk.splat(-1.0);
        const D xm = bk.up1(x, v0);
        const D PS = bk.scan_excl(x);
        const I rg = bk.bits3(modes_pk, ln);
        const D al = ra_l(rg), cl = rc_l(rg), bl = rb_l(rg);
        const D du = x - al * xm - cl;
        D bv = bk.splat(tol), brhs = bk.splat(0.0);
        I bid = bk.splati(-1);
        const Bm j1 = (ln >= 1) & valid;
#define HVP_CAND(T, OK, S, RHS)                                                           \
    {                                                                                     \
        const I id__ = ln + (T) * 12;                                                     \
        const D s__ = (S);                                                                \
        const Bm take__ = (OK) & (s__ > bv) & !bk.bit128(am_lo, am_hi, id__);             \
        bv = bk.sel(take__, s__, bv); bid = bk.seli(take__, id__, bid);                   \
        brhs = bk.sel(take__, (RHS), brhs);                                               \
    }
        HVP_CAND(T_UB, valid, x - ub, ub);
        HVP_CAND(T_LB, valid, lb - x, -lb);
        const D dv = x - xm;
        HVP_CAND(T_ACC, j1, dv - accmax, accmax);
        HVP_CAND(T_DEC, j1, decmin - dv, -decmin);
        {
            const Bm fx = j1 & (ln < L);
            HVP_CAND(T_UHI, fx, du - bl * P->umax, cl + bl * P->umax);
            HVP_CAND(T_ULO, fx, bl * P->umin - du, -(cl + bl * P->umin));
        }
        HVP_CAND(T_PHI, j1, PS - (P->pmax - pc), bk.splat(P->pmax - pc));
        HVP_CAND(T_PLO, j1, (P->pmin - pc) - PS, bk.splat(-(P->pmin - pc)));
        if (has_sf) {
            const D o = bk.sel(bk.bit32(satf, ln), NEG, bk.splat(1.0));
            HVP_CAND(T_SF, j1, o * (PS - sf), o * sf);
        }
        if (has_sb) {
            const D o = bk.sel(bk.bit32(satb, ln), NEG, bk.splat(1.0));
            HVP_CAND(T_SB, j1, o * (sb - PS), -(o * sb));
        }
#undef HVP_CAND
        double best_v;
        bk.gmax_arg(bv, bid, best_v, pid);
        if (pid < 0) {
            // ---- node solved: objective = tracking closed form + input cost + L1 penalties ----
            const D hoff_l = hw1 * ((double)(N - 1) - lnd) + hw2;
            const D hdiag_l = hw1 * ((double)(N - 1) - lnd) + hd;
            D term = x * (0.5 * hdiag_l * x + hoff_l * PS + gt);
            const D uu = bk.div(du, bl);
            term += bk.sel(ln < L, qu * uu * uu, bk.splat(0.0));
            if (has_sf) { const D s = PS - sf; term += bk.sel((ln >= 1) & (s > 0.0), ww * s, bk.splat(0.0)); }
            if (has_sb) { const D s = sb - PS; term += bk.sel((ln >= 1) & (s > 0.0), ww * s, bk.splat(0.0)); }
            node_done(0, ct + bk.gsum(bk.sel(valid, term, bk.splat(0.0))));
            return;
        }
        const int pt = pid / 12;
        pj = pid - 12 * pt;
        prhs = bk.bcast(brhs, pj);
        pcoef = 1.0;
        switch (pt) {
            case T_UB: pkind = 0; psgn = 1.0; break;
            case T_LB: pkind = 0; psgn = -1.0; break;
            case T_ACC: pkind = 1; psgn = 1.0; break;
            case T_DEC: pkind = 1; psgn = -1.0; break;
            case T_UHI: pkind = 1; psgn = 1.0; pcoef = ra(mode(pj)); break;
            case T_ULO: pkind = 1; psgn = -1.0; pcoef = ra(mode(pj)); break;
            case T_PHI: pkind = 2; psgn = 1.0; break;
            case T_PLO: pkind = 2; psgn = -1.0; break;
            case T_SF: pkind = 2; psgn = ((satf >> pj) & 1u) ? -1.0 : 1.0; break;
            default: pkind = 2; psgn = ((satb >> pj) & 1u) ? 1.0 : -1.0; break;
        }
        p_soft = pt >= T_SF;
        // n_p, H^-1 n_p and n_p'H^-1 n_p stay fixed while p is being added
        np = bk.splat(0.0); yp = bk.splat(0.0);
#pragma unroll
        for (int c = 0; c < G; ++c) {
            const double cc = coef_at(pkind, pj, psgn, pcoef, c);
            np = bk.sel(ln == c, bk.splat(cc), np);
            yp += hinv[c] * cc;
        }
        nHn = bk.gsum(np * yp);
        yps = bk.scan_excl(yp);
        lam_p = 0.0;
        state = S_STEP;
    }

    // ---- STEP: one primal-dual step towards adding p ----------------------------------------
    HVP_CD void do_step() {
        const double tol = 1e-9, ww = P->w;
        const I ln = bk.lane();
        if (++it > 40 * N + 60) { node_done(2, 0.0); return; }
        const double cp = bk.gsum(np * x) - prhs;
        // see flat_core.cuh: a row that reaches its boundary at the end of a partial step joins the active
        // set with its accumulated multiplier (zero-length full step)
        const bool zero_step = (cp <= tol);
        if (zero_step && !(lam_p > 0.0)) { state = S_SELECT; return; }
        // d_a = n_a' yp for slot a (lane a owns its row description);  r = Ginv d
        D d;
        {
            const D vj = bk.shfl(yp, s_j), vjm = bk.shfl(yp, s_j - 1), ps = bk.shfl(yps, s_j);
            d = s_sgn * bk.sel(s_kind == 0, vj, bk.sel(s_kind == 1, vj - s_coef * vjm, ps));
            d = bk.sel(ln < q, d, bk.splat(0.0));
        }
        D r = bk.splat(0.0);
#pragma unroll
        for (int b = 0; b < G; ++b) r += ginv[b] * bk.bcast(d, b);
        const double nz = nHn - bk.gsum(d * r);
        const bool dependent = (q == N) || !(nz > 1e-11 * nHn);
        const double INF = HUGE_VAL;
        if (zero_step && dependent) { node_done(2, 0.0); return; }
        const double t2 = dependent ? INF : (zero_step ? 0.0 : bk.sdiv(cp, nz));
        double t1, t3; int k1, k3;
        {
            const Bm act_ok = ln < q;
            const Bm pos = act_ok & (r > 1e-14);
            const D c1v = bk.sel(pos, bk.div(lam, bk.sel(pos, r, bk.splat(1.0))), bk.splat(INF));
            bk.gmin_arg(c1v, ln, t1, k1);
            const Bm softneg = act_ok & (r < -1e-14) & (s_id >= T_SF * 12);
            const D c3v = bk.sel(softneg, bk.div(ww - lam, bk.sel(softneg, -r, bk.splat(1.0))), bk.splat(INF));
            bk.gmin_arg(c3v, ln, t3, k3);
        }
        const double t3p = p_soft ? (ww - lam_p) : INF;
        const double t = fmin(fmin(t1, t2), fmin(t3, t3p));
        if (!(t < INF)) { node_done(1, 0.0); return; }          // infeasible node
        dual += t * cp - (dependent ? 0.0 : 0.5 * t * t * nz);  // dD/dt = violation of p along the step
        if (dual > inc) { node_done(1, 0.0); return; }          // the node cannot beat the incumbent
        double ru[G];
#pragma unroll
        for (int a = 0; a < G; ++a) ru[a] = bk.bcast(r, a);
        if (!dependent) {
            D z = yp;
#pragma unroll
            for (int a = 0; a < G; ++a) z -= Y[a] * ru[a];
            x -= t * z;
        }
        lam -= t * r;
        lam_p += t;
        if (t == t2) {
            // p becomes slot q: bordering update of Ginv with Schur complement nz
            const double is = bk.sdiv(1.0, nz);
            const Bm isq = ln == q;
#pragma unroll
            for (int b = 0; b < G; ++b) {
                D nb = ginv[b] + r * (ru[b] * is);
                nb = (b == q) ? -(r * is) : nb;
                nb = bk.sel(isq, bk.splat(b == q ? is : -ru[b] * is), nb);
                ginv[b] = (b <= q) ? nb : ginv[b];
            }
#pragma unroll
            for (int c = 0; c < G; ++c) Y[c] = (c == q) ? yp : Y[c];
            lam = bk.sel(isq, bk.splat(lam_p), lam);
            s_sgn = bk.sel(isq, bk.splat(psgn), s_sgn);
            s_coef = bk.sel(isq, bk.splat(pcoef), s_coef);
            s_kind = bk.seli(isq, bk.splati(pkind), s_kind);
            s_j = bk.seli(isq, bk.splati(pj), s_j);
            s_id = bk.seli(isq, bk.splati(pid), s_id);
            mark(pid, true);
            ++q;
            state = S_SELECT;
            return;
        }
        if (t == t3p) {                                          // soft p saturates: flip, not added
            if (pid / 12 == T_SF) satf ^= (1u << pj); else satb ^= (1u << pj);
            state = S_SELECT;
            return;
        }
        int drop;
        if (t == t1) drop = k1;
        else {                                                   // active soft row saturates: flip + drop
            drop = k3;
            const int id = bk.bcasti(s_id, drop), j = id % 12;
            if (id / 12 == T_SF) satf ^= (1u << j); else satb ^= (1u << j);
        }
        mark(bk.bcasti(s_id, drop), false);
        {   // Ginv <- Ginv - g_k g_k'/g_kk, delete row/column `drop`, compact slots
            D ck = bk.splat(0.0);
#pragma unroll
            for (int c = 0; c < G; ++c) ck = (c == drop) ? ginv[c] : ck;
            double rowk[G];
#pragma unroll
            for (int b = 0; b < G; ++b) rowk[b] = bk.bcast(ginv[b], drop);
            double gkk = 1.0;
#pragma unroll
            for (int b = 0; b < G; ++b) gkk = (b == drop) ? rowk[b] : gkk;
            const double ikk = bk.sdiv(1.0, gkk);
            const Bm mv = ln >= drop;
#pragma unroll
            for (int b = 0; b < G; ++b) ginv[b] -= ck * (rowk[b] * ikk);
#pragma unroll
            for (int b = 0; b < G; ++b) ginv[b] = bk.sel(mv, bk.dn1(ginv[b]), ginv[b]);   // rows up
#pragma unroll
            for (int b = 0; b + 1 < G; ++b) {                                             // columns left
                ginv[b] = (b >= drop) ? ginv[b + 1] : ginv[b];
                Y[b] = (b >= drop) ? Y[b + 1] : Y[b];
            }
            ginv[G - 1] = bk.splat(0.0); Y[G - 1] = bk.splat(0.0);
            lam = bk.sel(mv, bk.dn1(lam), lam);
            s_sgn = bk.sel(mv, bk.dn1(s_sgn), s_sgn);
            s_coef = bk.sel(mv, bk.dn1(s_coef), s_coef);
            s_kind = bk.seli(mv, bk.dn1i(s_kind), s_kind);
            s_j = bk.seli(mv, bk.dn1i(s_j), s_j);
            s_id = bk.seli(mv, bk.dn1i(s_id), s_id);
            --q;
            const Bm dead = ln >= q;                              // rows / columns beyond q stay zero
#pragma unroll
            for (int b = 0; b < G; ++b) ginv[b] = bk.sel(dead | (b >= q), bk.splat(0.0), ginv[b]);
        }
        // state stays S_STEP: continue with the same p
    }

    // ---- results -----------------------------------------------------------------------------
    HVP_CD LocalResult finish(double* u_out, double* x_out, int32_t* mode_out) {
        LocalResult R;
        R.nodes = nodes; R.qp_iters = iters;
        const I ln = bk.lane();
        const Bm valid = ln < N;
        const int np1 = N + 1;
        if ((sub_M > 1 ? own : inc) < HUGE_VAL) {
            R.obj = sub_M > 1 ? own : inc;
            R.status = timeout ? HVP_ST_TIME_LIMIT : limit ? HVP_ST_NODE_LIMIT : (trouble ? HVP_ST_NUMERIC : HVP_ST_OPTIMAL);
            const I rg = bk.bits3(best_modes, ln);
            const D vprev = bk.up1(best, v0);
            const D uu = (best - ra_l(rg) * vprev - rc_l(rg)) / rb_l(rg);
            const D pk = pc + bk.scan_excl(best);           // p_{j+1}
            bk.st(u_out, ln, uu, valid);
            bk.sti(mode_out, ln, rg, valid);
            bk.st(x_out, ln + 1, pk, valid);
            bk.st(x_out, ln + 1 + np1, best, valid);
            bk.st(x_out, ln, bk.splat(p0), ln == 0);
            bk.st(x_out, ln + np1, bk.splat(v0), ln == 0);
        } else {
            R.obj = HUGE_VAL;
            R.status = timeout ? HVP_ST_TIME_LIMIT : limit ? HVP_ST_NODE_LIMIT : (trouble ? HVP_ST_NUMERIC : HVP_ST_INFEASIBLE);
            bk.st(u_out, ln, bk.splat(0.0), valid);
            bk.sti(mode_out, ln, bk.splati(-1), valid);
            bk.st(x_out, ln + 1, bk.splat(0.0), valid);
            bk.st(x_out, ln + 1 + np1, bk.splat(0.0), valid);
            bk.st(x_out, ln, bk.splat(0.0), ln == 0);
            bk.st(x_out, ln + np1, bk.splat(0.0), ln == 0);
        }
        return R;
    }

    // one trip of the state machine (each block at most once, in pipeline order)
    HVP_CD void trip() {
        if (state == S_NEXT) do_next();
        if (state == S_BUILD) do_build();
        if (state == S_SELECT) do_select();
        if (state == S_STEP) do_step();
    }

    HVP_CD LocalResult solve(double* u_out, double* x_out, int32_t* mode_out) {
        begin();
        while (state != S_DONE) trip();
        return finish(u_out, x_out, mode_out);
    }
};

}  // namespace hvp
