// coord.cu -- fused coordinator glue of the switching ("g") ADMM controller (SURVEY.md 8f rank 1).
//
// One consensus round of fleet_g_admm.py:255-301 (+ the restated round logic of dmpcpwa's GAdmmCoordinator /
// dmpcrl's MpcAdmm, hybrid_vehicle_platoon_b200/fleet_g_admm.py) is, for every agent: solve the fixed-sequence QP
// (compiled-MPC kernel, one launch per role), then
//     z_j   <- mean of the copies of vehicle j's trajectory (own, the copy held by j+1, the copy held by j-1)
//     y     <- y + rho (copy - z)                         for the agent's own block and its neighbour copies
//     u_j   <- the QP's inputs where the QP was solved
//     seq_j <- PWA region sequence of the roll-out of u_j from the current state (the next round's fixed modes)
// and the next round's parameter vector [leader window | y blocks | z blocks].  As torch ops this was ~280 tiny
// launches per round (r02i launch list: 1.1 ms of a 2.1 ms round at 1024 scenarios x 15 vehicles); here it is ONE
// kernel, one thread per (scenario, vehicle): a vehicle's update needs only its neighbours' QP outputs, which it reads
// straight from the role buffers, recomputing the two neighbouring z's instead of synchronising.
//
// Arithmetic: every expression is evaluated in the order of the torch formulation with explicit round-to-nearest
// multiplies and adds (no FMA contraction), so the consensus variables are bit-identical to the unfused path
// (tests/test_gpu_sweep.py compares the two); only the per-scenario cost is summed in vehicle order.
#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>

#include "../../include/hvp.h"
#include "hvp_internal.h"

namespace hvp {

struct GRole {                    // one role = one compiled formulation = one launch (leader / last / interior)
    double* params;               // [count*S][npar]   next round's parameters (written here)
    double* x0;                   // [count*S][2]
    double* mass;                 // [count*S]
    int32_t* fm;                  // [count*S][N]      next round's fixed mode sequences
    const double* uo;             // [count*S][N]      QP outputs of the round just solved
    const double* xo;             // [count*S][2][N+1]
    const double* eo;             // [count*S][ne]     copies: front (if any) then back (if any), (2, N+1) each
    const double* ob;             // [count*S]
    const int32_t* st;            // [count*S]
    int first, count, npar, ne;
};

struct GArgs {
    int n, N, S, init;
    double rho, mug;
    double edge[6], cf[7], bg[7], dd[7];
    GRole role[3];                // 0: vehicle 0, 1: vehicle n-1, 2: vehicles 1..n-2 (count 0 when n == 2)
    const double* x;              // [S][n][2]    current state
    const double* mass;           // [S][n]
    const double* lwin;           // [S][2][N+1]  leader window
    double* y;                    // [S][n][3][2][N+1]  multipliers of the blocks (front copy, own, back copy)
    double* u;                    // [S][n][N]    current inputs (in: start / previous round; out: updated)
    double* tr;                   // [S][n][2][N+1]  PWA roll-out of u
    double* cost;                 // [S]
    uint8_t* ok;                  // [S]  and-accumulated over the rounds of a warm start (set to 1 by init)
};

__device__ __forceinline__ int role_of(const GArgs& A, int i) { return i == 0 ? 0 : (i == A.n - 1 ? 1 : 2); }

// QP outputs of vehicle j in scenario s
struct VOut {
    const double *uo, *xo, *cf, *cb;
    bool good;
    double ob;
};
__device__ __forceinline__ VOut vout(const GArgs& A, int s, int j) {
    const GRole& R = A.role[role_of(A, j)];
    const int64_t b = (int64_t)s * R.count + (j - R.first);
    const int np1 = A.N + 1;
    VOut o;
    o.uo = R.uo + b * A.N;
    o.xo = R.xo + b * 2 * np1;
    const double* e = R.eo + b * R.ne;
    o.cf = j > 0 ? e : nullptr;
    o.cb = j < A.n - 1 ? e + (j > 0 ? 2 * np1 : 0) : nullptr;
    o.good = R.st[b] == 2;
    o.ob = R.ob[b];
    return o;
}

// z of vehicle j, entry e of its (2, N+1) block: (own + copy held by j+1) + copy held by j-1, over the count
__device__ __forceinline__ double zval(const GArgs& A, int s, int j, int e) {
    const VOut me = vout(A, s, j);
    double acc = me.xo[e];
    double cnt = 1.0;
    if (j < A.n - 1) { acc = __dadd_rn(acc, vout(A, s, j + 1).cf[e]); cnt += 1.0; }
    if (j > 0) { acc = __dadd_rn(acc, vout(A, s, j - 1).cb[e]); cnt += 1.0; }
    return acc / cnt;
}

__global__ void __launch_bounds__(128)
gadmm_round_kernel(const __grid_constant__ GArgs A) {
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = A.n, N = A.N, np1 = N + 1, blk = 2 * np1;
    if (t >= (int64_t)A.S * n) return;
    const int s = (int)(t / n), j = (int)(t - (int64_t)s * n);
    const GRole& R = A.role[role_of(A, j)];
    const int64_t b = (int64_t)s * R.count + (j - R.first);
    double* yb = A.y + (size_t)t * 3 * blk;          // [front | own | back]
    double* uj = A.u + (size_t)t * N;
    double* trj = A.tr + (size_t)t * blk;
    const double m = A.mass[t];
    const double p0 = A.x[2 * t], v0 = A.x[2 * t + 1];

    if (!A.init) {
        // ---- inputs of the solved QPs, multiplier update with the new z ----
        const VOut me = vout(A, s, j);
        if (me.good)
            for (int k = 0; k < N; ++k) uj[k] = me.uo[k];
        for (int e = 0; e < blk; ++e) {
            const double zj = zval(A, s, j, e);
            yb[blk + e] = __dadd_rn(yb[blk + e], __dmul_rn(A.rho, __dadd_rn(me.xo[e], -zj)));
            if (j > 0) yb[e] = __dadd_rn(yb[e], __dmul_rn(A.rho, __dadd_rn(me.cf[e], -zval(A, s, j - 1, e))));
            if (j < n - 1)
                yb[2 * blk + e] = __dadd_rn(yb[2 * blk + e], __dmul_rn(A.rho, __dadd_rn(me.cb[e], -zval(A, s, j + 1, e))));
        }
    } else {
        for (int e = 0; e < 3 * blk; ++e) yb[e] = 0.0;
    }
    // ---- PWA roll-out of u_j from the current state: trajectory and region sequence ----
    {
        double p = p0, v = v0;
        trj[0] = p; trj[np1] = v;
        for (int k = 0; k < N; ++k) {
            int r = 0;
            for (int q = 0; q < 6; ++q) r += (A.edge[q] + 1e-9 < v) ? 1 : 0;      // bucketize(v, edges + 1e-9, right=False)
            R.fm[b * N + k] = r;
            const double a = __dadd_rn(1.0, (-A.cf[r]) / m);
            const double bb = A.bg[r] / m;
            const double c = __dadd_rn(-A.mug, -(A.dd[r] / m));
            const double pn = __dadd_rn(p, v);
            const double vn = __dadd_rn(__dadd_rn(__dmul_rn(a, v), __dmul_rn(bb, uj[k])), c);
            p = pn; v = vn;
            trj[k + 1] = p; trj[np1 + k + 1] = v;
        }
    }
    // ---- next round's parameters: [leader window | y blocks | z blocks], blocks = [front (j > 0), own, back (j < n-1)] ----
    double* P = R.params + (size_t)b * R.npar;
    R.x0[2 * b] = p0; R.x0[2 * b + 1] = v0;
    R.mass[b] = m;
    const double* lw = A.lwin + (size_t)s * blk;
    for (int e = 0; e < blk; ++e) P[e] = lw[e];
    int o = blk;
    if (j > 0) { for (int e = 0; e < blk; ++e) P[o + e] = yb[e]; o += blk; }
    for (int e = 0; e < blk; ++e) P[o + e] = yb[blk + e];
    o += blk;
    if (j < n - 1) { for (int e = 0; e < blk; ++e) P[o + e] = yb[2 * blk + e]; o += blk; }
    // z blocks.  init: z = the roll-out of the start inputs -- the neighbours' roll-outs are recomputed here (cheap)
    for (int d = -1; d <= 1; ++d) {
        const int jj = j + d;
        if (jj < 0 || jj >= n) continue;
        if (!A.init) {
            for (int e = 0; e < blk; ++e) P[o + e] = zval(A, s, jj, e);
        } else if (d == 0) {
            for (int e = 0; e < blk; ++e) P[o + e] = trj[e];
        } else {
            const int64_t tt = t + d;
            const double mm = A.mass[tt];
            const double* uu = A.u + (size_t)tt * N;
            double p = A.x[2 * tt], v = A.x[2 * tt + 1];
            P[o] = p; P[o + np1] = v;
            for (int k = 0; k < N; ++k) {
                int r = 0;
                for (int q = 0; q < 6; ++q) r += (A.edge[q] + 1e-9 < v) ? 1 : 0;
                const double a = __dadd_rn(1.0, (-A.cf[r]) / mm);
                const double bb = A.bg[r] / mm;
                const double c = __dadd_rn(-A.mug, -(A.dd[r] / mm));
                const double pn = __dadd_rn(p, v);
                const double vn = __dadd_rn(__dadd_rn(__dmul_rn(a, v), __dmul_rn(bb, uu[k])), c);
                p = pn; v = vn;
                P[o + k + 1] = p; P[o + np1 + k + 1] = v;
            }
        }
        o += blk;
    }
    // ---- per scenario: cost of the round (solved QPs only, vehicle order) and the and-accumulated status ----
    if (j == 0) {
        if (A.init) {
            A.ok[s] = 1; A.cost[s] = 0.0;
        } else {
            double c = 0.0;
            bool all = true;
            for (int i = 0; i < n; ++i) {
                const VOut vo = vout(A, s, i);
                if (vo.good) c = __dadd_rn(c, vo.ob); else all = false;
            }
            A.cost[s] = c;
            if (!all) A.ok[s] = 0;
        }
    }
}


// ---- decentralized / sequential controllers: constant-velocity extrapolation of every vehicle's neighbours and the
// leader-trajectory window of the timestep (fleet_decent_mld.py:329-331, :421-428) in one launch -------------------------
struct ObsArgs {
    int n, N, S, leader_index;
    long long lx_len, lx_sstride;     // leader trajectory: [S or 1][2][lx_len], scenario stride 0 when shared
    double ts;
    const double* x;                  // [S][n][2]
    const double* lx;
    const long long* t;               // device-side timestep index
    double *xf, *xb, *xl;             // [S][n][2][N+1] each
};
__global__ void __launch_bounds__(128)
decent_observe_kernel(const __grid_constant__ ObsArgs A) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = A.n, N = A.N, np1 = N + 1, blk = 2 * np1;
    if (tid >= (int64_t)A.S * n) return;
    const int s = (int)(tid / n), i = (int)(tid - (int64_t)s * n);
    // my own prediction is my back neighbour's x_front and my front neighbour's x_back
    double p = A.x[2 * tid];
    const double v = A.x[2 * tid + 1];
    double* f = i + 1 < n ? A.xf + (size_t)(tid + 1) * blk : nullptr;
    double* b = i > 0 ? A.xb + (size_t)(tid - 1) * blk : nullptr;
    for (int k = 0; k <= N; ++k) {
        if (f) { f[k] = p; f[np1 + k] = v; }
        if (b) { b[k] = p; b[np1 + k] = v; }
        p = __dadd_rn(p, __dmul_rn(A.ts, v));            // sequential sums, as the reference (p_{k+1} = p_k + ts v_k)
    }
    if (i == A.leader_index) {
        const long long t = *A.t;
        const double* l = A.lx + (size_t)s * A.lx_sstride;
        double* o = A.xl + (size_t)tid * blk;
        for (int k = 0; k <= N; ++k) { o[k] = l[t + k]; o[np1 + k] = l[A.lx_len + t + k]; }
    }
}

// ---- naive ADMM: z- and y-update of a consensus round and the next round's parameter vectors
// (fleet_naive_admm.py:421-468) in one launch, read straight from the role solves' outputs -------------------------------
// The same device code serves hvp_admm_round_dev (step = false: leader window from lwin, no statuses, no logs) and the
// three phases of hvp_admm_step_dev (step = true: t / r on the device, leader window from the trajectory, zeros for a
// solve that was not optimal, logs).
struct ARole {
    double* params;                   // [count*S][5 * 2(N+1)]: leader window | y_front | z_front | y_back | z_back
    double* x0;                       // [count*S][1][2]     (step PACK)
    const double* xo;                 // [count*S][2][N+1]   own prediction of the round just solved
    const double* eo;                 // [count*S][ne]       copies: x_front (if not front) then x_back (if not trailer)
    const double* u;                  // [count*S][N]        (step ADOPT)
    const int32_t *modes, *status, *nodes;   // step only; status NULL: every solve counts as optimal
    int count, ne, has_front, has_back;
};
struct AdmmArgs {
    int n, N, S, nroles, phase;       // phase: HVP_ADMM_PACK | HVP_ADMM_ROUND | HVP_ADMM_ADOPT
    bool step;
    double rho;
    ARole role[4];
    int role_of[64], local_of[64];    // vehicle -> role, index among the role's vehicles
    const double* lwin;               // hvp_admm_round_dev: [S][2][N+1]
    const long long* t;               // step: device timestep index
    const int32_t* r;                 // step: device round index
    const double *x, *lx;             // step: states [S][n][2], leader trajectory [S or 1][2][lx_len]
    long long lx_len, lx_sstride, T;
    int n_modes;
    int mode_gear[16];
    double *y_front, *y_back, *zf, *zb, *xs;   // [S][n][2][N+1] each
    int32_t *ND, *fa, *gear0, *ST;
    double *u0, *U;
};
__device__ __forceinline__ int64_t arow(const AdmmArgs& A, int s, int j) {
    return (int64_t)s * A.role[A.role_of[j]].count + A.local_of[j];
}
__device__ __forceinline__ bool aok(const ARole& R, int64_t b) { return !R.status || R.status[b] == HVP_OPTIMAL; }
// what vehicle j's solve contributes to the z-update: its own prediction and the copies it holds of its neighbours,
// all zero when the solve was not optimal (solve_mpc(raises=False) zeros x and the copies, LocalMpcADMM._post)
struct AOut { const double *own, *cf, *cb; bool ok; };
__device__ __forceinline__ AOut aout(const AdmmArgs& A, int s, int j) {
    AOut o = {nullptr, nullptr, nullptr, false};
    if (j < 0 || j >= A.n) return o;
    const ARole& R = A.role[A.role_of[j]];
    const int64_t b = arow(A, s, j);
    const int blk = 2 * (A.N + 1);
    o.own = R.xo + b * blk;
    const double* e = R.eo + b * R.ne;
    o.cf = R.has_front ? e : nullptr;
    o.cb = R.has_back ? e + (R.has_front ? blk : 0) : nullptr;
    o.ok = aok(R, b);
    return o;
}
__device__ __forceinline__ double aval(const double* p, bool ok, int e) { return ok ? p[e] : 0.0; }
// z of vehicle k (a, m, b: the outputs of vehicles k-1, k, k+1): (own + x_front copy held by k+1) / 2 at the front,
// (own + x_back copy held by k-1) / 2 at the rear, (own + both) / 3 inside -- in exactly this order of additions
// (fleet_naive_admm.py:421-447)
__device__ __forceinline__ double azval(int n, int k, const AOut& a, const AOut& m, const AOut& b, int e) {
    const double own = aval(m.own, m.ok, e);
    if (k == 0) return __dadd_rn(own, aval(b.cf, b.ok, e)) / 2.0;
    if (k == n - 1) return __dadd_rn(own, aval(a.cb, a.ok, e)) / 2.0;
    return __dadd_rn(__dadd_rn(own, aval(b.cf, b.ok, e)), aval(a.cb, a.ok, e)) / 3.0;
}
// entry e of the leader-window block: lwin, or leader_x[:, t : t+N+1] with columns past the end reading the last one
__device__ __forceinline__ double alwin(const AdmmArgs& A, int s, int e, long long t) {
    const int np1 = A.N + 1;
    if (!A.step) return A.lwin[(size_t)s * 2 * np1 + e];
    const int row = e / np1;
    long long c = t + (e - row * np1);
    c = c < 0 ? 0 : (c >= A.lx_len ? A.lx_len - 1 : c);
    return A.lx[(size_t)s * A.lx_sstride + row * A.lx_len + c];
}
__global__ void __launch_bounds__(128)
admm_round_kernel(const __grid_constant__ AdmmArgs A) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = A.n, N = A.N, np1 = N + 1, blk = 2 * np1;
    if (tid >= (int64_t)A.S * n) return;
    const int s = (int)(tid / n), j = (int)(tid - (int64_t)s * n);
    const ARole& R = A.role[A.role_of[j]];
    const int64_t b = arow(A, s, j);
    const long long t = A.step ? *A.t : 0;
    if (A.phase == HVP_ADMM_ADOPT) {  // first inputs of the last round, gears from the mode table, logs
        const bool ok = aok(R, b);
        const double u0 = ok ? R.u[b * N] : 0.0;
        A.u0[tid] = u0;
        int gear = 6;
        if (A.gear0) {
            if (ok) {
                int m = R.modes[b * N];
                m = m < 0 ? 0 : (m >= A.n_modes ? A.n_modes - 1 : m);
                gear = A.mode_gear[m];
            }
            A.gear0[tid] = gear;
        }
        if (t < 0 || t >= A.T) return;
        const size_t row = (size_t)t * A.S + s;
        double* Ur = A.U + row * (A.gear0 ? 2 * n : n);
        Ur[j] = u0;
        if (A.gear0) Ur[n + j] = (double)gear;
        A.ST[row * n + j] = R.status[b];
        return;
    }
    double* P = R.params + b * (5 * blk);
    const size_t o = (size_t)tid * blk;
    if (A.phase == HVP_ADMM_PACK) {
        if (A.step) {
            R.x0[2 * b] = A.x[2 * tid]; R.x0[2 * b + 1] = A.x[2 * tid + 1];
            if (t > 0) {              // the neighbours' previous predictions, shifted (fleet_naive_admm.py:392-402)
                for (int e = 0; e < blk; ++e) {
                    const int row = e / np1, k = e - row * np1, src = row * np1 + (k < N ? k + 1 : N);
                    if (j > 0) A.zf[o + e] = A.xs[o - blk + src];
                    if (j < n - 1) A.zb[o + e] = A.xs[o + blk + src];
                }
            }
        }
        for (int e = 0; e < blk; ++e) {
            P[e] = alwin(A, s, e, t); P[blk + e] = A.y_front[o + e]; P[2 * blk + e] = A.zf[o + e];
            P[3 * blk + e] = A.y_back[o + e]; P[4 * blk + e] = A.zb[o + e];
        }
        return;
    }
    AOut w[5];                        // vehicles j-2 .. j+2
    for (int d = 0; d < 5; ++d) w[d] = aout(A, s, j - 2 + d);
    const AOut& me = w[2];
    for (int e = 0; e < blk; ++e) {
        double yf = A.y_front[o + e], yb = A.y_back[o + e], zfv = A.zf[o + e], zbv = A.zb[o + e];
        A.xs[o + e] = aval(me.own, me.ok, e);
        if (j > 0) {                  // y_front += rho (x_front copy - z of the vehicle in front); next target z_{j-1}
            zfv = azval(n, j - 1, w[0], w[1], w[2], e);
            yf = __dadd_rn(yf, __dmul_rn(A.rho, __dadd_rn(aval(me.cf, me.ok, e), -zfv)));
        }
        if (j < n - 1) {
            zbv = azval(n, j + 1, w[2], w[3], w[4], e);
            yb = __dadd_rn(yb, __dmul_rn(A.rho, __dadd_rn(aval(me.cb, me.ok, e), -zbv)));
        }
        A.y_front[o + e] = yf; A.y_back[o + e] = yb; A.zf[o + e] = zfv; A.zb[o + e] = zbv;
        P[e] = alwin(A, s, e, t); P[blk + e] = yf; P[2 * blk + e] = zfv; P[3 * blk + e] = yb; P[4 * blk + e] = zbv;
    }
    // logs of the round.  ND: every vehicle's node count (a max: the same whatever the order).  failed_at: in the first
    // round of the episode the scenario's first thread resets the row and scans every vehicle; later, only a vehicle whose
    // solve failed looks at the vehicles before it, and the lowest failing one writes the row if it is still empty -- one
    // writer per scenario, and nothing beyond the atomic for the rounds in which every solve is optimal
    if (!A.step || t < 0 || t >= A.T) return;
    const int rr = *A.r;
    atomicMax(A.ND + (size_t)t * A.S + s, R.nodes[b]);
    int32_t* F = A.fa + 3 * (size_t)s;
    if (t == 0 && rr == 0) {
        if (j != 0) return;
        F[0] = -1; F[1] = -1; F[2] = 0;
        for (int i = 0; i < n; ++i) {
            const int st = A.role[A.role_of[i]].status[arow(A, s, i)];
            if (st != HVP_OPTIMAL) { F[0] = 0; F[1] = 0; F[2] = st; break; }
        }
        return;
    }
    if (me.ok) return;
    for (int i = 0; i < j; ++i)
        if (A.role[A.role_of[i]].status[arow(A, s, i)] != HVP_OPTIMAL) return;
    if (F[0] < 0) { F[0] = (int32_t)t; F[1] = rr; F[2] = R.status[b]; }
}

// ---- centralized controller: the leader window before the solve, the adoption of its answer after it
// (fleet_cent_mld.py:22-32, mpcs/mpc_gear.py:116-135) -------------------------------------------------------------
struct CentArgs {
    int n, N, S, phase, npar, n_modes;
    long long lx_len, lx_sstride, T;  // leader trajectory: [S or 1][2][lx_len], scenario stride 0 when shared
    int mode_gear[16];
    const long long* t;
    const double* lx;
    double* params;
    const double *u, *obj;
    const int32_t *modes, *status, *nodes;
    double* u0;
    int32_t* gear0;
    double *U, *objl;
    int32_t *stl, *ndl, *ab;
};
__global__ void __launch_bounds__(128)
cent_step_kernel(const __grid_constant__ CentArgs A) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = A.n, N = A.N, np1 = N + 1;
    if (tid >= (int64_t)A.S * n) return;
    const int s = (int)(tid / n), i = (int)(tid - (int64_t)s * n);
    const long long t = *A.t;
    if (A.phase == HVP_CENT_PACK) {
        // the scenario's n threads share the 2(N+1) entries of the window
        const double* l = A.lx + (size_t)s * A.lx_sstride;
        double* P = A.params + (size_t)s * A.npar;
        for (int e = i; e < 2 * np1; e += n) {
            const int row = e / np1, k = e - row * np1;
            long long c = t + k;
            c = c < 0 ? 0 : (c >= A.lx_len ? A.lx_len - 1 : c);
            P[e] = l[row * A.lx_len + c];
        }
        return;
    }
    const bool ok = A.status[s] == HVP_OPTIMAL;
    const double u0 = ok ? A.u[(size_t)tid * N] : 0.0;
    A.u0[tid] = u0;
    int gear = 6;
    if (A.gear0) {
        if (ok) {
            int m = A.modes[(size_t)tid * N];
            m = m < 0 ? 0 : (m >= A.n_modes ? A.n_modes - 1 : m);
            gear = A.mode_gear[m];
        }
        A.gear0[tid] = gear;
    }
    if (t < 0 || t >= A.T) return;
    const int w = A.gear0 ? 2 * n : n;
    double* Ur = A.U + ((size_t)t * A.S + s) * w;
    Ur[i] = u0;
    if (A.gear0) Ur[n + i] = (double)gear;
    if (i == 0) {
        const size_t r = (size_t)t * A.S + s;
        A.objl[r] = A.obj[s]; A.stl[r] = A.status[s]; A.ndl[r] = A.nodes[s];
        if (t == 0) A.ab[s] = ok ? -1 : 0;
        else if (!ok && A.ab[s] < 0) A.ab[s] = (int32_t)t;
    }
}

// ---- event-based controller: the glue of one iteration of TrackingEventBasedCoordinator.get_control and the end of a
// timestep (fleet_event_based.py:42-107) -------------------------------------------------------------------------------
struct EvArgs {
    hvp_event_iter g;
    int count[8];                     // agents of each group: a group's rows are [scenario][slot]
    long long lx_sstride;             // leader trajectory scenario stride, 0 when shared
};
// agent i optimises the members first..first + nl - 1 ([i-1, i, i+1] clipped at the ends; [0, 1] for both when n = 2)
__host__ __device__ __forceinline__ int ev_first(int n, int i) { return (n == 2 || i == 0) ? 0 : (i == n - 1 ? n - 2 : i - 1); }
__host__ __device__ __forceinline__ int ev_nmem(int n, int i) { return (n == 2 || i == 0 || i == n - 1) ? 2 : 3; }
__device__ __forceinline__ int64_t ev_row(const EvArgs& A, int s, int i) {
    return (int64_t)s * A.count[A.g.group_of[i]] + A.g.slot_of[i];
}

__global__ void __launch_bounds__(128)
event_pack_kernel(const __grid_constant__ EvArgs A) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = A.g.n, N = A.g.N, np1 = N + 1, blk = 2 * np1;
    if (tid >= (int64_t)A.g.S * n) return;
    const int s = (int)(tid / n), i = (int)(tid - (int64_t)s * n);
    const hvp_event_group& G = A.g.group[A.g.group_of[i]];
    const int64_t b = ev_row(A, s, i);
    const int nl = G.n_local, f = ev_first(n, i);
    for (int l = 0; l < nl; ++l) {
        const size_t src = (size_t)s * n + f + l, dst = (size_t)b * nl + l;
        G.x0[2 * dst] = A.g.x[2 * src]; G.x0[2 * dst + 1] = A.g.x[2 * src + 1];
        for (int e = 0; e < blk; ++e) G.xg[dst * blk + e] = A.g.SG[src * blk + e];
        for (int k = 0; k < N; ++k) G.ug[dst * N + k] = A.g.UG[src * N + k];
    }
    double* P = G.params + (size_t)b * G.n_param;
    if (G.has_leader) {
        const long long t = *A.g.t, L = A.g.leader_len;
        const double* l = A.g.leader_x + (size_t)s * A.lx_sstride;
        for (int e = 0; e < blk; ++e) {
            const int row = e / np1;
            long long c = t + (e - row * np1);
            c = c < 0 ? 0 : (c >= L ? L - 1 : c);
            P[e] = l[row * L + c];
        }
    } else {
        for (int e = 0; e < blk; ++e) P[e] = 0.0;
    }
    const double* f2 = i > 1 ? A.g.SG + ((size_t)s * n + i - 2) * blk : nullptr;
    const double* b2 = i < n - 2 ? A.g.SG + ((size_t)s * n + i + 2) * blk : nullptr;
    for (int e = 0; e < blk; ++e) {
        P[blk + e] = f2 ? f2[e] : 0.0;
        P[2 * blk + e] = b2 ? b2[e] : 0.0;
    }
}

// one warp per scenario
__global__ void __launch_bounds__(128)
event_select_kernel(const __grid_constant__ EvArgs A) {
    const int64_t w = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const int lane = threadIdx.x & 31;
    const int n = A.g.n, N = A.g.N, blk = 2 * (N + 1);
    if (w >= A.g.S) return;
    const int s = (int)w;
    if (!A.g.active[s]) return;
    constexpr int NONE = 1 << 30;
    constexpr unsigned FULL = 0xffffffffu;
    double best = -INFINITY;
    int bi = NONE, nd = INT32_MIN;
    bool feas = false;
    for (int i = lane; i < n; i += 32) {
        const hvp_event_group& G = A.g.group[A.g.group_of[i]];
        const int64_t b = ev_row(A, s, i);
        const double c1 = G.status[b] == HVP_OPTIMAL ? G.obj[b] : INFINITY;
        const double dec = __dadd_rn(G.cost[b], -c1);       // inf - inf = NaN: never > threshold
        feas |= (bool)isfinite(c1);
        nd = max(nd, G.nodes[b]);
        if (dec > A.g.threshold && (bi == NONE || dec > best)) { best = dec; bi = i; }
    }
    // largest decrease, the first agent among equal ones
    for (int o = 16; o > 0; o >>= 1) {
        const double ob = __shfl_xor_sync(FULL, best, o);
        const int oi = __shfl_xor_sync(FULL, bi, o);
        if (oi != NONE && (bi == NONE || ob > best || (ob == best && oi < bi))) { best = ob; bi = oi; }
        nd = max(nd, __shfl_xor_sync(FULL, nd, o));
    }
    feas = __any_sync(FULL, feas);
    const long long t = *A.g.t;
    if (lane == 0 && t >= 0 && t < A.g.T) {
        const size_t r = (size_t)t * A.g.S + s;
        if (!feas) A.g.FEAS[r] = 0;
        A.g.ND[r] = max(A.g.ND[r], nd);
        A.g.WIN[r * A.g.iters + A.g.it] = bi == NONE ? -1 : bi;
    }
    if (bi == NONE) {                 // nobody improved: the reference stops iterating this timestep
        if (lane == 0) A.g.active[s] = 0;
        return;
    }
    // the winner's plan overwrites the shared guesses of its members
    const hvp_event_group& G = A.g.group[A.g.group_of[bi]];
    const int64_t b = ev_row(A, s, bi);
    const int nl = G.n_local;
    const size_t base = (size_t)s * n + ev_first(n, bi);
    for (int e = lane; e < nl * blk; e += 32) {
        const int l = e / blk;
        A.g.SG[(base + l) * blk + (e - l * blk)] = G.x[(size_t)b * nl * blk + e];
    }
    for (int e = lane; e < nl * N; e += 32) {
        const int l = e / N;
        const size_t d = (base + l) * N + (e - l * N);
        A.g.UG[d] = G.u[(size_t)b * nl * N + e];
        if (A.g.GG) {
            int m = G.modes[(size_t)b * nl * N + e];
            m = m < 0 ? 0 : (m >= A.g.n_modes ? A.g.n_modes - 1 : m);
            A.g.GG[d] = A.g.mode_gear[m];
        }
    }
}

__global__ void __launch_bounds__(128)
event_adopt_kernel(const __grid_constant__ EvArgs A) {
    const int64_t tid = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int n = A.g.n, N = A.g.N, np1 = N + 1;
    if (tid >= (int64_t)A.g.S * n) return;
    const int s = (int)(tid / n), i = (int)(tid - (int64_t)s * n);
    double* sg = A.g.SG + (size_t)tid * 2 * np1;
    double* ug = A.g.UG + (size_t)tid * N;
    int32_t* gg = A.g.GG ? A.g.GG + (size_t)tid * N : nullptr;
    const double u0 = ug[0];
    A.g.u0[tid] = u0;
    if (gg) A.g.gear0[tid] = gg[0];
    const long long t = *A.g.t;
    if (t >= 0 && t < A.g.T) {
        double* Ur = A.g.U_log + ((size_t)t * A.g.S + s) * (gg ? 2 * n : n);
        Ur[i] = u0;
        if (gg) Ur[n + i] = (double)gg[0];
    }
    // shifted previous solution: drop column 0, repeat the last one (fleet_event_based.py:98-103)
    for (int k = 0; k < N; ++k) { sg[k] = sg[k + 1]; sg[np1 + k] = sg[np1 + k + 1]; }
    for (int k = 0; k + 1 < N; ++k) {
        ug[k] = ug[k + 1];
        if (gg) gg[k] = gg[k + 1];
    }
    if (i == 0) A.g.active[s] = 1;
}

}  // namespace hvp

using namespace hvp;

// hvp.h: hvp_gadmm_round_dev
extern "C" int hvp_gadmm_round_dev(hvp_ctx* c, const hvp_gadmm_round* g, void* stream) {
    if (!c || !g) return hvp_fail(-1, "gadmm_round: NULL argument");
    if (g->n < 2 || g->N < 1 || g->N > 16 || g->S < 0) return hvp_fail(-4, "gadmm_round: bad sizes (n=%d N=%d S=%d)", g->n, g->N, g->S);
    if (g->S == 0) return 0;
    if (!g->x || !g->mass || !g->lwin || !g->y || !g->u || !g->tr || !g->cost || !g->ok)
        return hvp_fail(-1, "gadmm_round: NULL array argument");
    GArgs A;
    A.n = g->n; A.N = g->N; A.S = g->S; A.init = g->init; A.rho = g->rho;
    A.mug = g->mug;
    for (int r = 0; r < 7; ++r) { A.cf[r] = g->cf[r]; A.bg[r] = g->bg[r]; A.dd[r] = g->dd[r]; }
    for (int q = 0; q < 6; ++q) A.edge[q] = g->edge[q];
    const int np1 = g->N + 1;
    for (int r = 0; r < 3; ++r) {
        const hvp_gadmm_role& s = g->role[r];
        GRole& R = A.role[r];
        R.first = r == 0 ? 0 : (r == 1 ? g->n - 1 : 1);
        R.count = r == 2 ? g->n - 2 : 1;
        const int na = (r == 2) ? 3 : 2;
        R.npar = (1 + 2 * na) * 2 * np1;
        R.ne = (na - 1) * 2 * np1;
        R.params = s.params; R.x0 = s.x0; R.mass = s.mass; R.fm = s.fixed_modes;
        R.uo = s.u; R.xo = s.x; R.eo = s.extra; R.ob = s.obj; R.st = s.status;
        if (R.count > 0 && (!R.params || !R.x0 || !R.mass || !R.fm || !R.uo || !R.xo || !R.eo || !R.ob || !R.st))
            return hvp_fail(-1, "gadmm_round: NULL role buffer (role %d)", r);
    }
    A.x = g->x; A.mass = g->mass; A.lwin = g->lwin; A.y = g->y; A.u = g->u; A.tr = g->tr; A.cost = g->cost; A.ok = g->ok;
    cudaError_t e = cudaSetDevice(c->device);
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "gadmm_round: cudaSetDevice: %s", cudaGetErrorString(e));
    cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
    const int64_t threads = (int64_t)g->S * g->n;
    gadmm_round_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, st>>>(A);
    e = cudaGetLastError();
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "gadmm_round: launch failed: %s", cudaGetErrorString(e));
    c->launches += 1;
    return 0;
}

// hvp.h: hvp_decent_observe_dev
extern "C" int hvp_decent_observe_dev(hvp_ctx* c, const hvp_decent_observe* g, void* stream) {
    if (!c || !g) return hvp_fail(-1, "decent_observe: NULL argument");
    if (g->n < 1 || g->N < 1 || g->S < 0 || g->leader_index < 0 || g->leader_index >= g->n)
        return hvp_fail(-4, "decent_observe: bad sizes (n=%d N=%d S=%d leader=%d)", g->n, g->N, g->S, g->leader_index);
    if (g->S == 0) return 0;
    if (!g->x || !g->leader_x || !g->t || !g->xf || !g->xb || !g->xl) return hvp_fail(-1, "decent_observe: NULL array argument");
    ObsArgs A;
    A.n = g->n; A.N = g->N; A.S = g->S; A.leader_index = g->leader_index; A.ts = g->ts;
    A.lx_len = g->leader_len; A.lx_sstride = g->leader_per_scenario ? 2 * g->leader_len : 0;
    A.x = g->x; A.lx = g->leader_x; A.t = (const long long*)g->t; A.xf = g->xf; A.xb = g->xb; A.xl = g->xl;
    cudaError_t e = cudaSetDevice(c->device);
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "decent_observe: cudaSetDevice: %s", cudaGetErrorString(e));
    cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
    const int64_t threads = (int64_t)g->S * g->n;
    decent_observe_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, st>>>(A);
    e = cudaGetLastError();
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "decent_observe: launch failed: %s", cudaGetErrorString(e));
    c->launches += 1;
    return 0;
}

// hvp.h: hvp_admm_round_dev
extern "C" int hvp_admm_round_dev(hvp_ctx* c, const hvp_admm_round* g, void* stream) {
    if (!c || !g) return hvp_fail(-1, "admm_round: NULL argument");
    if (g->n < 2 || g->n > 64 || g->N < 1 || g->S < 0 || g->nroles < 1 || g->nroles > 4)
        return hvp_fail(-4, "admm_round: bad sizes (n=%d N=%d S=%d roles=%d)", g->n, g->N, g->S, g->nroles);
    if (g->S == 0) return 0;
    if (!g->lwin || !g->y_front || !g->y_back || !g->zf || !g->zb || !g->xs) return hvp_fail(-1, "admm_round: NULL array argument");
    AdmmArgs A = {};
    A.n = g->n; A.N = g->N; A.S = g->S; A.nroles = g->nroles; A.rho = g->rho;
    A.phase = g->pack_only ? HVP_ADMM_PACK : HVP_ADMM_ROUND;
    const int blk = 2 * (g->N + 1);
    int counts[4] = {0, 0, 0, 0};
    for (int i = 0; i < g->n; ++i) {
        const int r = g->role_of[i];
        if (r < 0 || r >= g->nroles) return hvp_fail(-4, "admm_round: role_of[%d] = %d out of range", i, r);
        A.role_of[i] = r; A.local_of[i] = counts[r]++;
    }
    for (int r = 0; r < g->nroles; ++r) {
        const hvp_admm_role& s = g->role[r];
        ARole& R = A.role[r];
        R.params = s.params; R.xo = s.x; R.eo = s.extra; R.count = counts[r];
        R.has_front = s.has_front; R.has_back = s.has_back; R.ne = (s.has_front + s.has_back) * blk;
        if (counts[r] > 0 && (!R.params || !R.xo || (R.ne > 0 && !R.eo))) return hvp_fail(-1, "admm_round: NULL role buffer (role %d)", r);
    }
    // a vehicle reads the copies its neighbours hold of it: vehicle i > 0 must hold x_front, i < n-1 must hold x_back
    for (int i = 0; i < g->n; ++i) {
        const ARole& R = A.role[A.role_of[i]];
        if ((i > 0) != (R.has_front != 0) || (i < g->n - 1) != (R.has_back != 0))
            return hvp_fail(-4, "admm_round: role of vehicle %d does not match its position (front / trailer copies)", i);
    }
    A.lwin = g->lwin; A.y_front = g->y_front; A.y_back = g->y_back; A.zf = g->zf; A.zb = g->zb; A.xs = g->xs;
    cudaError_t e = cudaSetDevice(c->device);
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "admm_round: cudaSetDevice: %s", cudaGetErrorString(e));
    cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
    const int64_t threads = (int64_t)g->S * g->n;
    admm_round_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, st>>>(A);
    e = cudaGetLastError();
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "admm_round: launch failed: %s", cudaGetErrorString(e));
    c->launches += 1;
    return 0;
}

// hvp.h: hvp_admm_step_dev
extern "C" int hvp_admm_step_dev(hvp_ctx* c, const hvp_admm_step* g, void* stream) {
    if (!c || !g) return hvp_fail(-1, "admm_step: NULL argument");
    const int n = g->n, ph = g->phase;
    if (n < 2 || n > 64 || g->N < 1 || g->S < 0 || g->nroles < 1 || g->nroles > 4 || g->T < 0 ||
        (ph != HVP_ADMM_PACK && ph != HVP_ADMM_ROUND && ph != HVP_ADMM_ADOPT))
        return hvp_fail(-4, "admm_step: bad sizes (n=%d N=%d S=%d roles=%d T=%lld phase=%d)", n, g->N, g->S, g->nroles,
                        (long long)g->T, ph);
    if ((ph != HVP_ADMM_ADOPT && g->leader_len < 1) || (ph == HVP_ADMM_ADOPT && g->gear0 && (g->n_modes < 1 || g->n_modes > 16)))
        return hvp_fail(-4, "admm_step: bad sizes (leader_len=%lld n_modes=%d)", (long long)g->leader_len, g->n_modes);
    AdmmArgs A = {};
    A.n = n; A.N = g->N; A.S = g->S; A.nroles = g->nroles; A.rho = g->rho; A.phase = ph; A.step = true;
    const int blk = 2 * (g->N + 1);
    int counts[4] = {0, 0, 0, 0};
    for (int i = 0; i < n; ++i) {
        const int r = g->role_of[i];
        if (r < 0 || r >= g->nroles) return hvp_fail(-4, "admm_step: role_of[%d] = %d out of range", i, r);
        A.role_of[i] = r; A.local_of[i] = counts[r]++;
    }
    for (int r = 0; r < g->nroles; ++r) {
        const hvp_admm_step_role& s = g->role[r];
        ARole& R = A.role[r];
        R.params = s.params; R.x0 = s.x0; R.xo = s.x; R.eo = s.extra; R.u = s.u; R.modes = s.modes; R.status = s.status;
        R.nodes = s.nodes; R.count = counts[r];
        R.has_front = s.has_front; R.has_back = s.has_back; R.ne = (s.has_front + s.has_back) * blk;
    }
    // a vehicle reads the copies its neighbours hold of it: vehicle i > 0 must hold x_front, i < n-1 must hold x_back
    for (int i = 0; i < n; ++i) {
        const ARole& R = A.role[A.role_of[i]];
        if ((i > 0) != (R.has_front != 0) || (i < n - 1) != (R.has_back != 0))
            return hvp_fail(-4, "admm_step: role of vehicle %d does not match its position (front / trailer copies)", i);
    }
    if (g->S == 0) return 0;
    if (!g->t || !g->y_front || !g->y_back || !g->zf || !g->zb || !g->xs ||
        (ph == HVP_ADMM_PACK && (!g->x || !g->leader_x)) ||
        (ph == HVP_ADMM_ROUND && (!g->r || !g->leader_x || !g->ND || !g->failed_at)) ||
        (ph == HVP_ADMM_ADOPT && (!g->u0 || !g->U_log || !g->ST)))
        return hvp_fail(-1, "admm_step: NULL array argument (phase %d)", ph);
    for (int r = 0; r < g->nroles; ++r) {
        const ARole& R = A.role[r];
        if (R.count == 0) continue;
        if ((ph == HVP_ADMM_PACK && (!R.params || !R.x0)) ||
            (ph == HVP_ADMM_ROUND && (!R.params || !R.xo || (R.ne > 0 && !R.eo) || !R.status || !R.nodes)) ||
            (ph == HVP_ADMM_ADOPT && (!R.u || !R.status || (g->gear0 && !R.modes))))
            return hvp_fail(-1, "admm_step: NULL role buffer (role %d, phase %d)", r, ph);
    }
    A.t = (const long long*)g->t; A.r = g->r; A.x = g->x; A.lx = g->leader_x;
    A.lx_len = g->leader_len; A.lx_sstride = g->leader_per_scenario ? 2 * g->leader_len : 0; A.T = g->T;
    A.n_modes = g->n_modes;
    for (int m = 0; m < 16; ++m) A.mode_gear[m] = g->mode_gear[m];
    A.y_front = g->y_front; A.y_back = g->y_back; A.zf = g->zf; A.zb = g->zb; A.xs = g->xs;
    A.ND = g->ND; A.fa = g->failed_at; A.u0 = g->u0; A.gear0 = g->gear0; A.U = g->U_log; A.ST = g->ST;
    cudaError_t e = cudaSetDevice(c->device);
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "admm_step: cudaSetDevice: %s", cudaGetErrorString(e));
    cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
    const int64_t threads = (int64_t)g->S * n;
    admm_round_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, st>>>(A);
    e = cudaGetLastError();
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "admm_step: launch failed: %s", cudaGetErrorString(e));
    c->launches += 1;
    return 0;
}

// hvp.h: hvp_cent_step_dev
extern "C" int hvp_cent_step_dev(hvp_ctx* c, const hvp_cent_step* g, void* stream) {
    if (!c || !g) return hvp_fail(-1, "cent_step: NULL argument");
    if (g->n < 1 || g->N < 1 || g->S < 0 ||
        (g->phase != HVP_CENT_PACK && g->phase != HVP_CENT_ADOPT))
        return hvp_fail(-4, "cent_step: bad sizes (n=%d N=%d S=%d phase=%d)", g->n, g->N, g->S, g->phase);
    CentArgs A;
    A.n = g->n; A.N = g->N; A.S = g->S; A.phase = g->phase; A.npar = g->n_param; A.n_modes = g->n_modes;
    A.lx_len = g->leader_len; A.lx_sstride = g->leader_per_scenario ? 2 * g->leader_len : 0; A.T = g->T;
    A.t = (const long long*)g->t; A.lx = g->leader_x; A.params = g->params;
    A.u = g->u; A.obj = g->obj; A.modes = g->modes; A.status = g->status; A.nodes = g->nodes;
    A.u0 = g->u0; A.gear0 = g->gear0; A.U = g->U_log; A.objl = g->obj_log; A.stl = g->status_log; A.ndl = g->nodes_log;
    A.ab = g->aborted_at;
    if (g->phase == HVP_CENT_PACK) {
        if (g->n_param < 2 * (g->N + 1) || g->leader_len < 1)
            return hvp_fail(-4, "cent_step: bad sizes (n_param=%d leader_len=%lld, N=%d)", g->n_param, (long long)g->leader_len, g->N);
        if (g->S == 0) return 0;
        if (!g->t || !g->leader_x || !g->params) return hvp_fail(-1, "cent_step: NULL array argument (pack)");
    } else {
        if (g->T < 0 || (g->gear0 && (g->n_modes < 1 || g->n_modes > 16)))
            return hvp_fail(-4, "cent_step: bad sizes (T=%lld n_modes=%d)", (long long)g->T, g->n_modes);
        if (g->S == 0) return 0;
        if (!g->t || !g->u || !g->obj || !g->status || !g->nodes || !g->u0 || !g->U_log || !g->obj_log || !g->status_log ||
            !g->nodes_log || !g->aborted_at || (g->gear0 && !g->modes))
            return hvp_fail(-1, "cent_step: NULL array argument (adopt)");
        for (int m = 0; m < 16; ++m) A.mode_gear[m] = g->mode_gear[m];
    }
    cudaError_t e = cudaSetDevice(c->device);
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "cent_step: cudaSetDevice: %s", cudaGetErrorString(e));
    cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
    const int64_t threads = (int64_t)g->S * g->n;
    cent_step_kernel<<<(unsigned)((threads + 127) / 128), 128, 0, st>>>(A);
    e = cudaGetLastError();
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "cent_step: launch failed: %s", cudaGetErrorString(e));
    c->launches += 1;
    return 0;
}

// hvp.h: hvp_event_iter_dev
extern "C" int hvp_event_iter_dev(hvp_ctx* c, const hvp_event_iter* g, void* stream) {
    if (!c || !g) return hvp_fail(-1, "event_iter: NULL argument");
    const int n = g->n, ph = g->phase;
    if (n < 2 || n > 64 || g->N < 1 || g->S < 0 || (ph != HVP_EVENT_PACK && ph != HVP_EVENT_SELECT && ph != HVP_EVENT_ADOPT))
        return hvp_fail(-4, "event_iter: bad sizes (n=%d N=%d S=%d phase=%d)", n, g->N, g->S, ph);
    if (g->ngroups < 1 || g->ngroups > 8 || g->iters < 1 || g->it < 0 || g->it >= g->iters || g->T < 0 ||
        (g->GG && (g->n_modes < 1 || g->n_modes > 16)))
        return hvp_fail(-4, "event_iter: bad sizes (groups=%d it=%d iters=%d T=%lld n_modes=%d)", g->ngroups, g->it, g->iters,
                        (long long)g->T, g->n_modes);
    EvArgs A;
    A.g = *g;
    uint64_t seen[8] = {0, 0, 0, 0, 0, 0, 0, 0};
    for (int r = 0; r < 8; ++r) A.count[r] = 0;
    for (int i = 0; i < n; ++i) {
        const int r = g->group_of[i], k = g->slot_of[i];
        if (r < 0 || r >= g->ngroups || k < 0 || k >= 64 || (seen[r] >> k & 1))
            return hvp_fail(-4, "event_iter: agent %d has group %d slot %d (out of range or taken)", i, r, k);
        if (g->group[r].n_local != ev_nmem(n, i))
            return hvp_fail(-4, "event_iter: group %d has %d members per agent, agent %d has %d", r, g->group[r].n_local, i,
                            ev_nmem(n, i));
        seen[r] |= 1ull << k;
        A.count[r] += 1;
    }
    for (int i = 0; i < n; ++i)       // the slots of a group are 0 .. count - 1
        if (g->slot_of[i] >= A.count[g->group_of[i]])
            return hvp_fail(-4, "event_iter: agent %d has slot %d of a group of %d", i, g->slot_of[i], A.count[g->group_of[i]]);
    bool lead = false;
    for (int r = 0; r < g->ngroups; ++r) {
        if (A.count[r] == 0) continue;
        const hvp_event_group& G = g->group[r];
        lead |= G.has_leader != 0;
        if (ph == HVP_EVENT_PACK && G.n_param < 6 * (g->N + 1))
            return hvp_fail(-4, "event_iter: group %d n_param=%d < 6(N+1)", r, G.n_param);
    }
    if (ph == HVP_EVENT_PACK && lead && g->leader_len < 1)
        return hvp_fail(-4, "event_iter: bad sizes (leader_len=%lld)", (long long)g->leader_len);
    if (g->S == 0) return 0;
    if (!g->t || !g->SG || !g->UG) return hvp_fail(-1, "event_iter: NULL array argument");
    for (int r = 0; r < g->ngroups; ++r) {
        const hvp_event_group& G = g->group[r];
        if (A.count[r] == 0) continue;
        if (ph == HVP_EVENT_PACK && (!G.x0 || !G.xg || !G.ug || !G.params))
            return hvp_fail(-1, "event_iter: NULL group buffer (pack, group %d)", r);
        if (ph == HVP_EVENT_SELECT && (!G.cost || !G.u || !G.x || !G.obj || !G.status || !G.nodes || (g->GG && !G.modes)))
            return hvp_fail(-1, "event_iter: NULL group buffer (select, group %d)", r);
    }
    if ((ph == HVP_EVENT_PACK && (!g->x || (lead && !g->leader_x))) ||
        (ph == HVP_EVENT_SELECT && (!g->active || !g->WIN || !g->FEAS || !g->ND)) ||
        (ph == HVP_EVENT_ADOPT && (!g->active || !g->U_log || !g->u0 || (g->GG && !g->gear0))))
        return hvp_fail(-1, "event_iter: NULL array argument (phase %d)", ph);
    A.lx_sstride = g->leader_per_scenario ? 2 * g->leader_len : 0;
    cudaError_t e = cudaSetDevice(c->device);
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "event_iter: cudaSetDevice: %s", cudaGetErrorString(e));
    cudaStream_t st = stream ? (cudaStream_t)stream : c->stream;
    const int64_t threads = (int64_t)g->S * (ph == HVP_EVENT_SELECT ? 32 : n);
    const unsigned blocks = (unsigned)((threads + 127) / 128);
    if (ph == HVP_EVENT_PACK) event_pack_kernel<<<blocks, 128, 0, st>>>(A);
    else if (ph == HVP_EVENT_SELECT) event_select_kernel<<<blocks, 128, 0, st>>>(A);
    else event_adopt_kernel<<<blocks, 128, 0, st>>>(A);
    e = cudaGetLastError();
    if (e != cudaSuccess) return hvp_fail(-100 - (int)e, "event_iter: launch failed: %s", cudaGetErrorString(e));
    c->launches += 1;
    return 0;
}
