// scalar_solver.h -- the FIRST-GENERATION per-thread MIQP solver (one problem per thread, nested data-dependent loops;
// r01a ncu: 5.8 of 32 lanes active).  TEST INFRASTRUCTURE ONLY: it is a second, independently written implementation of
// the velocity-space branch and bound that tests/test_host_core.py runs against the oracle and against the product's
// cores (coop_core.cuh, flat_core.cuh) on the host.  The product library does not contain it any more (round 2).
#pragma once
#include "../../hybrid_vehicle_platoon_b200/csrc/miqp_core.cuh"

namespace hvp {

template <int NMAX>
struct LocalLayout {
    static constexpr int TRI = NMAX * (NMAX + 1) / 2;
    static constexpr int O_HINV = 0;             // packed lower H^-1
    static constexpr int O_GINV = TRI;           // packed lower (N'H^-1N)^-1 of the active set
    static constexpr int O_X = 2 * TRI;
    static constexpr int O_LAM = O_X + NMAX;
    static constexpr int O_D = O_LAM + NMAX;
    static constexpr int O_R = O_D + NMAX;
    static constexpr int O_YP = O_R + NMAX;      // H^-1 n_p, later reused for w = n_p - N r
    static constexpr int O_GT = O_YP + NMAX;     // tracking gradient
    static constexpr int O_LB = O_GT + NMAX;
    static constexpr int O_UB = O_LB + NMAX;
    static constexpr int O_SF = O_UB + NMAX;     // soft rows PS_j <= sf[j]
    static constexpr int O_SB = O_SF + NMAX;     // soft rows PS_j >= sb[j]
    static constexpr int O_BEST = O_SB + NMAX;   // incumbent velocities
    static constexpr int O_XSTAR = O_BEST + NMAX;
    static constexpr int O_RLO = O_XSTAR + NMAX + 1;
    static constexpr int O_RHI = O_RLO + NMAX + 1;
    static constexpr int SIZE = O_RHI + NMAX + 1;  // doubles per thread
};

// decoded structured row:  n = sgn * base,  base = e_j | e_j - a e_{j-1} | sum_{i<j} e_i
struct Row {
    int kind;      // 0 single, 1 difference, 2 prefix sum
    int j;
    double sgn, a, rhs;
};

template <int NMAX, int ST>
struct LocalSolver {
    using LY = LocalLayout<NMAX>;
    double* W;                         // this thread's strided work array
    const LocalParams* P;
    int N, flags;
    double p0, v0, pc;                 // pc = p_1 = p0 + v0 (ts = 1)
    double inv_m, a_lo, a_hi, c_lo, c_hi;   // region dynamics (regions 0-3 / 4-6)
    double hw1, hw2, hd;               // tracking Hessian closed form
    double ct;                         // tracking constant (incl. k = 0,1 slack penalties)
    bool has_sf, has_sb;
    bool notrack;                               // no reference term (setup)
    int L;                             // stages 0..L-1 have fixed regions
    uint64_t modes_pk;                 // 3 bits per stage
    uint64_t act_lo, act_hi;           // active constraint ids (8 bits each: t*12 + j)
    uint64_t am_lo, am_hi;             // active-set membership bitmap, bit t*12 + j
    uint32_t satf, satb;               // soft rows currently in "violated" orientation
    int q, iters;

    HVP_HD double& w(int off, int i) const { return W[(size_t)(off + i) * ST]; }
    HVP_HD static int tri(int i, int j) { return i >= j ? i * (i + 1) / 2 + j : j * (j + 1) / 2 + i; }
    HVP_HD double ra(int rg) const { return rg < 4 ? a_lo : a_hi; }
    HVP_HD double rc(int rg) const { return rg < 4 ? c_lo : c_hi; }
    HVP_HD double rb(int rg) const { return P->bgear[rg] * inv_m; }
    HVP_HD int mode(int k) const { return (int)((modes_pk >> (3 * k)) & 7u); }
    HVP_HD void set_mode(int k, int rg) {
        modes_pk = (modes_pk & ~(7ull << (3 * k))) | ((uint64_t)rg << (3 * k));
    }
    HVP_HD int act(int a) const { return (int)(((a < 8 ? act_lo >> (8 * a) : act_hi >> (8 * (a - 8)))) & 0xffu); }
    HVP_HD void set_act(int a, int id) {
        if (a < 8) act_lo = (act_lo & ~(0xffull << (8 * a))) | ((uint64_t)id << (8 * a));
        else act_hi = (act_hi & ~(0xffull << (8 * (a - 8)))) | ((uint64_t)id << (8 * (a - 8)));
    }
    HVP_HD bool is_active(int id) const { return id < 64 ? (am_lo >> id) & 1u : (am_hi >> (id - 64)) & 1u; }
    HVP_HD void mark(int id, bool on) {
        if (id < 64) am_lo = on ? (am_lo | (1ull << id)) : (am_lo & ~(1ull << id));
        else am_hi = on ? (am_hi | (1ull << (id - 64))) : (am_hi & ~(1ull << (id - 64)));
    }
    HVP_HD double Hoff(int j) const { return hw1 * (double)(N - 1 - j) + hw2; }
    HVP_HD double Hdiag(int j) const { return hw1 * (double)(N - 1 - j) + hd; }

    // -------------------------------------------------------------------------------------
    HVP_HD void setup(double* W_, const LocalParams* P_, int flags_, double mass, const double* x0,
                      const double* xf, const double* xb, const double* xl) {
        W = W_; P = P_; N = P->N; flags = flags_;
        p0 = x0[0]; v0 = x0[1]; pc = p0 + v0;
        inv_m = 1.0 / mass;                         // models.py:447-473 + forward_euler (ts = 1)
        a_lo = 1.0 - P->c1 * inv_m; a_hi = 1.0 - P->c2 * inv_m;
        c_lo = -P->mug; c_hi = -P->mug - P->dfr * inv_m;
        const bool is_front = flags & 1, is_leader = flags & 2, is_trailer = flags & 4;
        // tracking terms  wp*(p_k + tau*v_k - Pk)^2 + wvv*(v_k - Vk)^2
        //   front  (fleet_decent_mld.py:110-121): tau = t0, Pk = pf_k - d0,           Vk = vf_k
        //   back   (:122-133):                    tau = 0,  Pk = pb_k + t0*vb_k + d0, Vk = vb_k
        //   leader (:134-141):                    tau = 0,  Pk = pl_k,                Vk = vl_k
        const bool tf = !is_front && !is_leader, tb = !is_trailer && !is_leader, tl = is_leader;
        const double wp = P->qxp, wvv = P->qxv, t0 = P->t0, d0 = P->d0;
        const int np1 = N + 1;
        const double nterm = (tf ? 1.0 : 0.0) + (tb ? 1.0 : 0.0) + (tl ? 1.0 : 0.0);
        // H_t[i][j] (i<j) = 2wp*(nterm*(N-1-j) + sum tau);  diag: 2wp*(nterm*(N-1-j) + sum tau^2) + 2wv*nterm
        hw1 = 2.0 * wp * nterm;
        hw2 = 2.0 * wp * (tf ? t0 : 0.0);
        hd = 2.0 * wp * (tf ? t0 * t0 : 0.0) + 2.0 * wvv * nterm;
        notrack = nterm < 0.5;     // no reference term: the Hessian is singular until every stage is fixed
        for (int j = 0; j < N; ++j) w(LY::O_GT, j) = 0.0;
        ct = 0.0;
        // rho_k = pc - Pk (k>=1);  g[j] = 2wp*(sum_{k>j+1} rho_k + tau*rho_{j+1}) - 2wv*V_{j+1}
        for (int kind = 0; kind < 3; ++kind) {
            const double* ref = kind == 0 ? xf : (kind == 1 ? xb : xl);
            const bool on = kind == 0 ? tf : (kind == 1 ? tb : tl);
            if (!on) continue;
            const double tau = kind == 0 ? t0 : 0.0;
            double suffix = 0.0;
            for (int k = N; k >= 0; --k) {
                const double pk = ref[k], vk = ref[np1 + k];
                const double Pk = (kind == 0) ? (pk - d0) : (kind == 1) ? (pk + t0 * vk + d0) : pk;
                if (k >= 1) {
                    const double rho = pc - Pk;
                    w(LY::O_GT, k - 1) += 2.0 * wp * (suffix + tau * rho) - 2.0 * wvv * vk;
                    ct += wp * rho * rho + wvv * vk * vk;
                    suffix += rho;
                } else {   // k = 0 terms are constants but count in objVal
                    const double e0 = p0 + tau * v0 - Pk, e1 = v0 - vk;
                    ct += wp * e0 * e0 + wvv * e1 * e1;
                }
            }
        }
        // soft safe-distance rows (fleet_decent_mld.py:191-208); k = 0,1 are constants
        has_sf = !is_front; has_sb = !is_trailer;
        const double ww = P->w, ds = P->d_safe;
        if (has_sf) {
            const double s0 = p0 - (xf[0] - ds), s1 = pc - (xf[1] - ds);
            ct += ww * (s0 > 0 ? s0 : 0.0) + ww * (s1 > 0 ? s1 : 0.0);
            for (int j = 1; j < N; ++j) w(LY::O_SF, j) = xf[j + 1] - ds - pc;
        }
        if (has_sb) {
            const double s0 = (xb[0] + ds) - p0, s1 = (xb[1] + ds) - pc;
            ct += ww * (s0 > 0 ? s0 : 0.0) + ww * (s1 > 0 ? s1 : 0.0);
            for (int j = 1; j < N; ++j) w(LY::O_SB, j) = xb[j + 1] + ds - pc;
        }
    }

    // -------------------------------------------------------------------------------------
    HVP_HD Row decode(int id) const {
        const int t = id / 12, j = id - 12 * t;
        Row r; r.j = j; r.a = 1.0;
        switch (t) {
            case T_UB: r.kind = 0; r.sgn = 1.0; r.rhs = w(LY::O_UB, j); break;
            case T_LB: r.kind = 0; r.sgn = -1.0; r.rhs = -w(LY::O_LB, j); break;
            case T_ACC: r.kind = 1; r.sgn = 1.0; r.rhs = P->a_acc - j * P->tight; break;
            case T_DEC: r.kind = 1; r.sgn = -1.0; r.rhs = -(P->a_dec + j * P->tight); break;
            case T_UHI: { const int rg = mode(j); r.kind = 1; r.sgn = 1.0; r.a = ra(rg); r.rhs = rc(rg) + rb(rg) * P->umax; } break;
            case T_ULO: { const int rg = mode(j); r.kind = 1; r.sgn = -1.0; r.a = ra(rg); r.rhs = -(rc(rg) + rb(rg) * P->umin); } break;
            case T_PHI: r.kind = 2; r.sgn = 1.0; r.rhs = P->pmax - pc; break;
            case T_PLO: r.kind = 2; r.sgn = -1.0; r.rhs = -(P->pmin - pc); break;
            case T_SF: { const double o = ((satf >> j) & 1u) ? -1.0 : 1.0; r.kind = 2; r.sgn = o; r.rhs = o * w(LY::O_SF, j); } break;
            default:   { const double o = ((satb >> j) & 1u) ? -1.0 : 1.0; r.kind = 2; r.sgn = -o; r.rhs = -o * w(LY::O_SB, j); } break;
        }
        return r;
    }
    // n' vec  (vec in the work array at offset off)
    HVP_HD double row_dot(const Row& r, int off) const {
        double s;
        if (r.kind == 0) s = w(off, r.j);
        else if (r.kind == 1) s = w(off, r.j) - r.a * w(off, r.j - 1);
        else { s = 0.0; for (int i = 0; i < r.j; ++i) s += w(off, i); }
        return r.sgn * s;
    }
    // vec += coef * n
    HVP_HD void row_axpy(const Row& r, double coef, int off) const {
        const double c = coef * r.sgn;
        if (r.kind == 0) w(off, r.j) += c;
        else if (r.kind == 1) { w(off, r.j) += c; w(off, r.j - 1) -= c * r.a; }
        else for (int i = 0; i < r.j; ++i) w(off, i) += c;
    }
    // out = H^-1 n
    HVP_HD void hinv_row(const Row& r, int off_out) const {
        for (int i = 0; i < N; ++i) {
            double s;
            if (r.kind == 0) s = w(LY::O_HINV, tri(i, r.j));
            else if (r.kind == 1) s = w(LY::O_HINV, tri(i, r.j)) - r.a * w(LY::O_HINV, tri(i, r.j - 1));
            else { s = 0.0; for (int k = 0; k < r.j; ++k) s += w(LY::O_HINV, tri(i, k)); }
            w(off_out, i) = r.sgn * s;
        }
    }

    // -------------------------------------------------------------------------------------
    // Build + solve the QP of the current node (modes 0..L-1 fixed). Returns 0 optimal,
    // 1 infeasible, 2 numeric/iteration trouble.  On success x (O_X) and *obj are set.
    HVP_HD int solve_node(double* obj) {
        const double tol = 1e-9;
        const double qu = P->qu, ww = P->w;
        // ---- Hessian (packed lower, built in the O_HINV area) and gradient (in O_D) ----
        for (int i = 0; i < N; ++i) {
            for (int j = 0; j < i; ++j) w(LY::O_HINV, tri(i, j)) = Hoff(i);
            w(LY::O_HINV, tri(i, i)) = Hdiag(i);
            w(LY::O_D, i) = w(LY::O_GT, i);
        }
        {   // stage 0 (x_{-1} = v0 is a constant): u_0 = (x_0 - (a v0 + c))/b
            const int rg = mode(0);
            const double ib = 1.0 / rb(rg), k0 = (ra(rg) * v0 + rc(rg)) * ib;
            w(LY::O_HINV, tri(0, 0)) += 2.0 * qu * ib * ib;
            w(LY::O_D, 0) += -2.0 * qu * k0 * ib;
        }
        for (int k = 1; k < L; ++k) {   // u_k = (x_k - a x_{k-1} - c)/b
            const int rg = mode(k);
            const double ib = 1.0 / rb(rg), ea = -ra(rg) * ib, kc = -rc(rg) * ib;
            w(LY::O_HINV, tri(k, k)) += 2.0 * qu * ib * ib;
            w(LY::O_HINV, tri(k - 1, k - 1)) += 2.0 * qu * ea * ea;
            w(LY::O_HINV, tri(k, k - 1)) += 2.0 * qu * ea * ib;
            w(LY::O_D, k) += 2.0 * qu * kc * ib;
            w(LY::O_D, k - 1) += 2.0 * qu * kc * ea;
        }
        // ---- in-place: Cholesky L, L^-1, then H^-1 = L^-T L^-1 (all packed lower) ----
        for (int j = 0; j < N; ++j) {
            double dd = w(LY::O_HINV, tri(j, j));
            for (int k = 0; k < j; ++k) { const double l = w(LY::O_HINV, tri(j, k)); dd -= l * l; }
            if (!(dd > 0.0)) return 2;
            dd = sqrt(dd);
            w(LY::O_HINV, tri(j, j)) = dd;
            const double inv = 1.0 / dd;
            for (int i = j + 1; i < N; ++i) {
                double s = w(LY::O_HINV, tri(i, j));
                for (int k = 0; k < j; ++k) s -= w(LY::O_HINV, tri(i, k)) * w(LY::O_HINV, tri(j, k));
                w(LY::O_HINV, tri(i, j)) = s * inv;
            }
        }
        for (int j = 0; j < N; ++j) {            // column j of L^-1 overwrites column j of L
            const double djj = 1.0 / w(LY::O_HINV, tri(j, j));
            w(LY::O_HINV, tri(j, j)) = djj;
            for (int i = j + 1; i < N; ++i) {
                double s = 0.0;
                for (int k = j; k < i; ++k) s += w(LY::O_HINV, tri(i, k)) * w(LY::O_HINV, tri(k, j));
                w(LY::O_YP, i) = -s / w(LY::O_HINV, tri(i, i));
                // store below after the loop over k used old L(i,k), k<i (columns > j untouched yet)
                w(LY::O_HINV, tri(i, j)) = w(LY::O_YP, i);
            }
        }
        for (int i = 0; i < N; ++i)              // (i,0..i): diagonal last -> safe in place
            for (int j = 0; j <= i; ++j) {
                double s = 0.0;
                for (int k = i; k < N; ++k) s += w(LY::O_HINV, tri(k, i)) * w(LY::O_HINV, tri(k, j));
                w(LY::O_HINV, tri(i, j)) = s;
            }
        for (int i = 0; i < N; ++i) {
            double s = 0.0;
            for (int j = 0; j < N; ++j) s -= w(LY::O_HINV, tri(i, j)) * w(LY::O_D, j);
            w(LY::O_X, i) = s;
        }
        q = 0; satf = 0; satb = 0; act_lo = act_hi = 0; am_lo = am_hi = 0;
        const int maxit = 40 * N + 60;
        int it = 0;

        for (;;) {
            // ---- most violated row (structured scan, prefix sums on the fly) ----
            double best = tol; int pid = -1;
            double PS = 0.0;
#define HVP_CAND(T, J, S)                                                     \
    {                                                                         \
        const double s__ = (S);                                               \
        if (s__ > best && !is_active((T) * 12 + (J))) { best = s__; pid = (T) * 12 + (J); } \
    }
            for (int j = 0; j < N; ++j) {
                const double xv = w(LY::O_X, j);
                HVP_CAND(T_UB, j, xv - w(LY::O_UB, j));
                HVP_CAND(T_LB, j, w(LY::O_LB, j) - xv);
                if (j >= 1) {
                    const double xm = w(LY::O_X, j - 1);
                    const double dv = xv - xm;
                    HVP_CAND(T_ACC, j, dv - (P->a_acc - j * P->tight));
                    HVP_CAND(T_DEC, j, (P->a_dec + j * P->tight) - dv);
                    if (j < L) {
                        const int rg = mode(j);
                        const double du = xv - ra(rg) * xm - rc(rg), bb = rb(rg);
                        HVP_CAND(T_UHI, j, du - bb * P->umax);
                        HVP_CAND(T_ULO, j, bb * P->umin - du);
                    }
                    HVP_CAND(T_PHI, j, PS - (P->pmax - pc));
                    HVP_CAND(T_PLO, j, (P->pmin - pc) - PS);
                    if (has_sf) {
                        const double s = PS - w(LY::O_SF, j);
                        HVP_CAND(T_SF, j, ((satf >> j) & 1u) ? -s : s);
                    }
                    if (has_sb) {
                        const double s = w(LY::O_SB, j) - PS;
                        HVP_CAND(T_SB, j, ((satb >> j) & 1u) ? -s : s);
                    }
                }
                PS += xv;
            }
#undef HVP_CAND
            if (pid < 0) break;
            const bool p_soft = pid >= T_SF * 12;
            double lam_p = 0.0;
            for (;;) {
                if (++it > maxit) { iters += it; return 2; }
                const Row rp = decode(pid);
                const double cp = row_dot(rp, LY::O_X) - rp.rhs;
                const bool zero_step = (cp <= tol);             // see flat_core.cuh: zero-length full step
                if (zero_step && !(lam_p > 0.0)) break;
                hinv_row(rp, LY::O_YP);                         // yp = H^-1 n_p
                const double nHn = row_dot(rp, LY::O_YP);
                // d = N' yp ; r = Ginv d ; nz = nHn - d'r
                for (int a = 0; a < q; ++a) w(LY::O_D, a) = row_dot(decode(act(a)), LY::O_YP);
                double nz = nHn;
                for (int a = 0; a < q; ++a) {
                    double s = 0.0;
                    for (int b = 0; b < q; ++b) s += w(LY::O_GINV, tri(a, b)) * w(LY::O_D, b);
                    w(LY::O_R, a) = s;
                    nz -= s * w(LY::O_D, a);
                }
                const bool dependent = (q == N) || !(nz > 1e-11 * nHn);
                const double INF = HUGE_VAL;
                if (zero_step && dependent) { iters += it; return 2; }
                const double t2 = dependent ? INF : (zero_step ? 0.0 : cp / nz);
                double t1 = INF, t3 = INF;
                int k1 = -1, k3 = -1;
                for (int a = 0; a < q; ++a) {
                    const double ra_ = w(LY::O_R, a);
                    if (ra_ > 1e-14) {
                        const double t = w(LY::O_LAM, a) / ra_;
                        if (t < t1) { t1 = t; k1 = a; }
                    } else if (ra_ < -1e-14 && act(a) >= T_SF * 12) {
                        const double t = (ww - w(LY::O_LAM, a)) / (-ra_);
                        if (t < t3) { t3 = t; k3 = a; }
                    }
                }
                const double t3p = p_soft ? (ww - lam_p) : INF;
                const double t = fmin(fmin(t1, t2), fmin(t3, t3p));
                if (!(t < INF)) { iters += it; return 1; }   // infeasible node
                if (!dependent) {
                    // w = n_p - N r (into O_YP), x -= t * H^-1 w
                    for (int i = 0; i < N; ++i) w(LY::O_YP, i) = 0.0;
                    row_axpy(rp, 1.0, LY::O_YP);
                    for (int a = 0; a < q; ++a) row_axpy(decode(act(a)), -w(LY::O_R, a), LY::O_YP);
                    for (int i = 0; i < N; ++i) {
                        double s = 0.0;
                        for (int j = 0; j < N; ++j) s += w(LY::O_HINV, tri(i, j)) * w(LY::O_YP, j);
                        w(LY::O_X, i) -= t * s;
                    }
                }
                for (int a = 0; a < q; ++a) w(LY::O_LAM, a) -= t * w(LY::O_R, a);
                lam_p += t;
                if (t == t2) {
                    // full step: p joins the active set; bordering update of Ginv with s = nz
                    const double is = 1.0 / nz;
                    for (int a = 0; a < q; ++a) {
                        const double ra_ = w(LY::O_R, a);
                        for (int b = 0; b <= a; ++b) w(LY::O_GINV, tri(a, b)) += ra_ * w(LY::O_R, b) * is;
                        w(LY::O_GINV, tri(q, a)) = -ra_ * is;
                    }
                    w(LY::O_GINV, tri(q, q)) = is;
                    set_act(q, pid); w(LY::O_LAM, q) = lam_p;
                    mark(pid, true);
                    ++q;
                    break;
                }
                if (t == t3p) {                     // soft p saturates before becoming feasible
                    const int j = pid % 12;
                    if (pid / 12 == T_SF) satf ^= (1u << j); else satb ^= (1u << j);
                    break;
                }
                int drop;
                if (t == t1) drop = k1;
                else {                               // active soft row saturates: flip + drop
                    drop = k3;
                    const int id = act(drop), j = id % 12;
                    if (id / 12 == T_SF) satf ^= (1u << j); else satb ^= (1u << j);
                }
                mark(act(drop), false);
                {   // Ginv <- Ginv - g_k g_k'/g_kk, then delete row/column `drop`
                    const double ikk = 1.0 / w(LY::O_GINV, tri(drop, drop));
                    for (int a = 0; a < q; ++a) w(LY::O_D, a) = w(LY::O_GINV, tri(a, drop));
                    for (int a = 0; a < q; ++a) {
                        if (a == drop) continue;
                        const int an = a > drop ? a - 1 : a;
                        for (int b = 0; b <= a; ++b) {
                            if (b == drop) continue;
                            const int bn = b > drop ? b - 1 : b;
                            w(LY::O_GINV, tri(an, bn)) =
                                w(LY::O_GINV, tri(a, b)) - w(LY::O_D, a) * w(LY::O_D, b) * ikk;
                        }
                    }
                }
                for (int a = drop; a + 1 < q; ++a) {
                    set_act(a, act(a + 1));
                    w(LY::O_LAM, a) = w(LY::O_LAM, a + 1);
                }
                --q;
            }
        }
        iters += it;
        // ---- objective at x: tracking closed form + input cost of fixed stages + L1 penalties ----
        double f = ct;
        {
            double PS = 0.0, vprev = v0;
            for (int j = 0; j < N; ++j) {
                const double xv = w(LY::O_X, j);
                f += xv * (0.5 * Hdiag(j) * xv + Hoff(j) * PS + w(LY::O_GT, j));
                if (j < L) {
                    const int rg = mode(j);
                    const double uu = (xv - ra(rg) * vprev - rc(rg)) / rb(rg);
                    f += qu * uu * uu;
                }
                if (j >= 1) {
                    if (has_sf) { const double s = PS - w(LY::O_SF, j); if (s > 0) f += ww * s; }
                    if (has_sb) { const double s = w(LY::O_SB, j) - PS; if (s > 0) f += ww * s; }
                }
                PS += xv; vprev = xv;
            }
        }
        *obj = f;
        return 0;
    }

    HVP_HD static int cand_get(uint64_t lo, uint64_t hi, int lv) {
        const unsigned sh = (unsigned)(7 * (lv < 9 ? lv : lv - 9));
        return (int)(((lv < 9 ? lo : hi) >> sh) & 0x7fu);
    }
    HVP_HD static void cand_set(uint64_t& lo, uint64_t& hi, int lv, int val) {
        const unsigned sh = (unsigned)(7 * (lv < 9 ? lv : lv - 9));
        uint64_t& t = lv < 9 ? lo : hi;
        t = (t & ~(0x7full << sh)) | ((uint64_t)val << sh);
    }

    // -------------------------------------------------------------------------------------
    // Branch and bound.  Outputs: u[N], xtraj[(2)(N+1)] row-major, mode_out[N].
    HVP_HD LocalResult solve(double* u_out, double* x_out, int32_t* mode_out) {
        LocalResult R;
        R.obj = HUGE_VAL; R.status = HVP_ST_INFEASIBLE; R.nodes = 0; R.qp_iters = 0;
        iters = 0; modes_pk = 0;
        double inc = HUGE_VAL;
        uint64_t best_modes = 0;
        uint64_t cand_lo = 0, cand_hi = 0;          // 7 candidate bits per level (levels 0..8 | 9..12)
        const double eps = 1e-9;
        bool trouble = false, limit = false;
#define HVP_CAND_GET(lv) cand_get(cand_lo, cand_hi, (lv))
#define HVP_CAND_SET(lv, val) cand_set(cand_lo, cand_hi, (lv), (val))
        int lev = 0;
        w(LY::O_RLO, 0) = v0; w(LY::O_RHI, 0) = v0; w(LY::O_XSTAR, 0) = v0;
        {
            int c0 = 0;
            for (int rg = 0; rg < NREG; ++rg)
                if (v0 >= P->edge[rg] && v0 <= P->edge[rg + 1]) c0 |= (1 << rg);
            HVP_CAND_SET(0, c0);
        }
        for (;;) {
            int cset = HVP_CAND_GET(lev);
            if (cset == 0) {
                if (lev == 0) break;
                --lev;
                continue;
            }
            // candidate region nearest to the parent's relaxed velocity
            int rg = -1; double bd = HUGE_VAL;
            const double xs = w(LY::O_XSTAR, lev);
            for (int c = 0; c < NREG; ++c) {
                if (!((cset >> c) & 1)) continue;
                const double lo = P->edge[c], hi = P->edge[c + 1];
                const double dist = xs < lo ? lo - xs : (xs > hi ? xs - hi : 0.0);
                if (dist < bd) { bd = dist; rg = c; }
            }
            cset &= ~(1 << rg);
            HVP_CAND_SET(lev, cset);
            set_mode(lev, rg);
            // reachable interval of v_{lev+1} through region rg (provable pruning only)
            const double jlo = fmax(w(LY::O_RLO, lev), P->edge[rg]), jhi = fmin(w(LY::O_RHI, lev), P->edge[rg + 1]);
            if (jlo > jhi + eps) continue;
            double nlo = fmax(ra(rg) * jlo + rc(rg) + rb(rg) * P->umin, jlo + P->a_dec + lev * P->tight);
            double nhi = fmin(ra(rg) * jhi + rc(rg) + rb(rg) * P->umax, jhi + P->a_acc - lev * P->tight);
            nlo = fmax(nlo, P->vmin); nhi = fmin(nhi, P->vmax);
            if (nlo > nhi + eps) continue;
            w(LY::O_RLO, lev + 1) = nlo - eps; w(LY::O_RHI, lev + 1) = nhi + eps;
            L = lev + 1;
            // merged simple bounds: state box (k>=1), region of fixed stages k=1..L-1 (x_{k-1}),
            // stage-0 accel and input rows (both bounds on x_0 = v_1)
            for (int j = 0; j < N; ++j) { w(LY::O_LB, j) = P->vmin; w(LY::O_UB, j) = P->vmax; }
            for (int k = 1; k < L; ++k) {
                w(LY::O_LB, k - 1) = fmax(w(LY::O_LB, k - 1), P->edge[mode(k)]);
                w(LY::O_UB, k - 1) = fmin(w(LY::O_UB, k - 1), P->edge[mode(k) + 1]);
            }
            {
                const int r0 = mode(0);
                w(LY::O_LB, 0) = fmax(w(LY::O_LB, 0), fmax(v0 + P->a_dec, ra(r0) * v0 + rc(r0) + rb(r0) * P->umin));
                w(LY::O_UB, 0) = fmin(w(LY::O_UB, 0), fmin(v0 + P->a_acc, ra(r0) * v0 + rc(r0) + rb(r0) * P->umax));
            }
            // p_1 = pc is a constant: its state rows are a feasibility check
            if (pc > P->pmax + eps || pc < P->pmin - eps) continue;
            if (notrack && L < N) {                         // only leaves are solved (enumeration, as the oracle)
                ++lev;
                w(LY::O_XSTAR, lev) = w(LY::O_XSTAR, lev - 1);
                int cn = 0;
                for (int c = 0; c < NREG; ++c)
                    if (P->edge[c] <= w(LY::O_RHI, lev) && P->edge[c + 1] >= w(LY::O_RLO, lev)) cn |= (1 << c);
                HVP_CAND_SET(lev, cn);
                continue;
            }
            double obj;
            const int st = solve_node(&obj);
            ++R.nodes;
            if (st == 2) { trouble = true; continue; }
            if (st == 1) continue;
            if (inc < HUGE_VAL && !(obj < inc - 1e-9 * fmax(1.0, fabs(inc)))) continue;   // bound
            if (L == N) {                                   // leaf: new incumbent
                inc = obj;
                for (int j = 0; j < N; ++j) w(LY::O_BEST, j) = w(LY::O_X, j);
                best_modes = modes_pk;
                continue;
            }
            if (P->max_nodes > 0 && R.nodes >= P->max_nodes) { limit = true; break; }
            ++lev;
            w(LY::O_XSTAR, lev) = w(LY::O_X, lev - 1);       // relaxed v_lev
            int cn = 0;
            for (int c = 0; c < NREG; ++c)
                if (P->edge[c] <= w(LY::O_RHI, lev) && P->edge[c + 1] >= w(LY::O_RLO, lev)) cn |= (1 << c);
            HVP_CAND_SET(lev, cn);
        }
#undef HVP_CAND_GET
#undef HVP_CAND_SET
        R.qp_iters = iters;
        const int np1 = N + 1;
        if (inc < HUGE_VAL) {
            R.obj = inc;
            R.status = limit ? HVP_ST_NODE_LIMIT : (trouble ? HVP_ST_NUMERIC : HVP_ST_OPTIMAL);
            double p = p0, v = v0;
            x_out[0] = p; x_out[np1] = v;
            for (int k = 0; k < N; ++k) {
                const int rg = (int)((best_modes >> (3 * k)) & 7u);
                const double vn = w(LY::O_BEST, k);
                u_out[k] = (vn - ra(rg) * v - rc(rg)) / rb(rg);
                mode_out[k] = rg;
                p = p + v; v = vn;
                x_out[k + 1] = p; x_out[np1 + k + 1] = v;
            }
        } else {
            R.status = limit ? HVP_ST_NODE_LIMIT : (trouble ? HVP_ST_NUMERIC : HVP_ST_INFEASIBLE);
            for (int k = 0; k < N; ++k) { u_out[k] = 0.0; mode_out[k] = -1; }
            for (int k = 0; k <= N; ++k) { x_out[k] = 0.0; x_out[np1 + k] = 0.0; }
        }
        return R;
    }
};

}  // namespace hvp
