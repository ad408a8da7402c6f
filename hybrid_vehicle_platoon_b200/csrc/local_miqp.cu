// local_miqp.cu -- batched per-vehicle hybrid-MPC MIQPs on sm_100a.
//
// Replaces the Gurobi solve behind LocalMpcMld.solve_mpc (fleet_decent_mld.py:21-223 /
// fleet_seq_mld.py:21-234 via dmpcpwa MpcMld.solve_mpc).
//
//   coop_miqp_kernel<G>  (default): a group of G = 8 (N <= 8) or 16 lanes solves one MIQP
//       cooperatively, all state in registers, warp shuffles for the reductions (coop_core.cuh).
//       The node QPs have 4..12 variables -- far too small for a CTA -- so a warp carries 4 (or 2)
//       independent branch-and-bound trees and the batch (scenario x vehicle x ADMM round)
//       fills the grid.
//   flat_miqp_kernel<N>  (batches >= 8192): one problem per lane, persistent warps (flat_core.cuh).
//   (The first design -- one thread per MIQP with nested loops, 5.8 of 32 lanes active -- left the library in
//   round 2; it survives as a second implementation for the host tests, tests/host_harness/scalar_solver.h.)
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>
#include <string.h>

#include "coop_core.cuh"
#include "flat_core.cuh"
#include "hvp_internal.h"
#include "miqp_core.cuh"

namespace hvp {

template <int G>
__global__ void __launch_bounds__(COOP_BLOCK)
coop_miqp_kernel(const __grid_constant__ LocalParams P, int64_t batch, const int32_t* __restrict__ flags,
                 const double* __restrict__ mass, const double* __restrict__ x0,
                 const double* __restrict__ xf, const double* __restrict__ xb,
                 const double* __restrict__ xl, double* __restrict__ u, double* __restrict__ x,
                 int32_t* __restrict__ modes, double* __restrict__ obj, int32_t* __restrict__ status,
                 int32_t* __restrict__ nodes, int32_t* __restrict__ qp_iters, int spread) {
    // packed: 32 / G problems per warp (throughput).  spread: ONE problem per warp, lanes G.. idle -- the groups of
    // a warp run different trees and serialise each other (r01m ncu: 15 of 32 lanes active), which is what a small
    // latency-critical batch (one scenario-timestep = n MIQPs) must not pay for
    const int64_t t = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (spread && (threadIdx.x & 31) >= G) return;
    const int64_t i = spread ? (t >> 5) : t / G;                              // problem of this group
    if (i >= batch) return;                                                   // whole group leaves
    const int N = P.N;
    const size_t S = 2 * (size_t)(N + 1);
    CoopSolver<DevBK<G>> sol;
    sol.setup(&P, flags[i], mass[i], x0 + 2 * i, xf ? xf + S * i : nullptr, xb ? xb + S * i : nullptr,
              xl ? xl + S * i : nullptr);
    const LocalResult R = sol.solve(u + (size_t)N * i, x + S * i, modes + (size_t)N * i);
    if (sol.bk.ln == 0) {
        obj[i] = R.obj;
        status[i] = R.status;
        nodes[i] = R.nodes;
        if (qp_iters) qp_iters[i] = R.qp_iters;
    }
}

// Latency path: ONE tree searched by M workers (one warp each, G lanes cooperating), see CoopSolver::sub_M.  Worker
// results go to scratch rows; the worker that finishes last (atomic count) keeps the best and writes the outputs.
// Scratch (per launch, armed by one 0xFF memset): done[batch] u32 counting up from 0xFFFFFFFF, keys[batch] u64 (0xFF..
// decodes to NaN = "no incumbent"), then batch x M result rows.
constexpr int COOP_SPLIT_MAX = 64;      // problems per launch that get several workers each
constexpr int COOP_SPLIT_ROW = 48;      // doubles per result row: u[N] x[2(N+1)] modes[N as double] obj status nodes iters

template <int G>
__global__ void __launch_bounds__(32)
coop_split_kernel(const __grid_constant__ LocalParams P, int64_t batch, int M, const int32_t* __restrict__ flags,
                  const double* __restrict__ mass, const double* __restrict__ x0,
                  const double* __restrict__ xf, const double* __restrict__ xb,
                  const double* __restrict__ xl, double* __restrict__ u, double* __restrict__ x,
                  int32_t* __restrict__ modes, double* __restrict__ obj, int32_t* __restrict__ status,
                  int32_t* __restrict__ nodes, int32_t* __restrict__ qp_iters, unsigned* __restrict__ done,
                  unsigned long long* __restrict__ keys, double* __restrict__ rows) {
    if (threadIdx.x >= G) return;
    const int64_t i = blockIdx.x / M;
    const int w = blockIdx.x % M;
    const int N = P.N, np1 = N + 1;
    const size_t S = 2 * (size_t)np1;
    CoopSolver<DevBK<G>> sol;
    sol.setup(&P, flags[i], mass[i], x0 + 2 * i, xf ? xf + S * i : nullptr, xb ? xb + S * i : nullptr,
              xl ? xl + S * i : nullptr);
    sol.sub_M = M; sol.sub_w = w; sol.shared = keys + i;
    double* row = rows + ((size_t)i * M + w) * COOP_SPLIT_ROW;
    int32_t* rmodes = reinterpret_cast<int32_t*>(row + N + S);             // N int32 in the space of N doubles
    const LocalResult R = sol.solve(row, row + N, rmodes);
    const int ln = sol.bk.ln;
    unsigned old = 0;
    if (ln == 0) {
        double* tail = row + 2 * N + S;
        tail[0] = R.obj; tail[1] = (double)R.status; tail[2] = (double)R.nodes; tail[3] = (double)R.qp_iters;
    }
    __syncwarp((1u << G) - 1u);
    __threadfence();
    if (ln == 0) old = atomicAdd(done + i, 1u);
    old = __shfl_sync((1u << G) - 1u, old, 0);
    if (old != (unsigned)(M - 2)) return;                     // not the last worker of this tree
    __threadfence();
    // ---- merge: best objective (lowest worker on ties), summed work, worst status ----
    double bv = HUGE_VAL;
    int bw = 0, nsum = 0, isum = 0;
    bool numeric = false, limited = false, timed = false;
    for (int c = 0; c < M; ++c) {
        const double* t = rows + ((size_t)i * M + c) * COOP_SPLIT_ROW + 2 * N + S;
        const double o = *reinterpret_cast<const volatile double*>(t);
        const int st = (int)*reinterpret_cast<const volatile double*>(t + 1);
        nsum += (int)*reinterpret_cast<const volatile double*>(t + 2);
        isum += (int)*reinterpret_cast<const volatile double*>(t + 3);
        if (o < bv) { bv = o; bw = c; }
        numeric = numeric || st == HVP_ST_NUMERIC; limited = limited || st == HVP_ST_NODE_LIMIT;
        timed = timed || st == HVP_ST_TIME_LIMIT;
    }
    const double* src = rows + ((size_t)i * M + bw) * COOP_SPLIT_ROW;
    const int32_t* smodes = reinterpret_cast<const int32_t*>(src + N + S);
    for (int e = ln; e < N; e += G) { u[(size_t)N * i + e] = src[e]; modes[(size_t)N * i + e] = smodes[e]; }
    for (int e = ln; e < (int)S; e += G) x[S * i + e] = src[N + e];
    if (ln == 0) {
        obj[i] = bv;
        status[i] = timed ? HVP_ST_TIME_LIMIT : limited ? HVP_ST_NODE_LIMIT
                          : (numeric ? HVP_ST_NUMERIC : (bv < HUGE_VAL ? HVP_ST_OPTIMAL : HVP_ST_INFEASIBLE));
        nodes[i] = nsum;
        if (qp_iters) qp_iters[i] = isum;
    }
}

// Persistent flat-state-machine kernel: one warp per CTA, one problem per lane, each warp owns a
// contiguous share of the batch and a lane that finishes refills from that share at once.
// STEAL = false compiles the sub-tree adoption of the launch tail OUT (about 900 SASS instructions): the kernel is bound
// by instruction fetch, and code that is never executed still spreads the hot loop over more cache lines.
template <int N, bool STEAL, bool HINTS>
// resident CTAs per SM are set by the shared-memory slab (10 at N = 6); telling the compiler lets it use the registers
// that occupancy leaves free instead of spilling
__global__ void __launch_bounds__(32, (N <= 6 ? 10 : (N == 7 ? 7 : (N == 8 ? 6 : 5))))
flat_miqp_kernel(const __grid_constant__ LocalParams P, int64_t batch, const int32_t* __restrict__ flags,
                 const double* __restrict__ mass, const double* __restrict__ x0,
                 const double* __restrict__ xf, const double* __restrict__ xb,
                 const double* __restrict__ xl, double* __restrict__ u, double* __restrict__ x,
                 int32_t* __restrict__ modes, double* __restrict__ obj, int32_t* __restrict__ status,
                 int32_t* __restrict__ nodes, int32_t* __restrict__ qp_iters, unsigned long long* __restrict__ counter,
                 double* __restrict__ scratch) {
    extern __shared__ double smem[];
    using Solver = FlatSolver<N, 32, false, HINTS>;
    const int lane = threadIdx.x;
    const size_t S = 2 * (size_t)(N + 1);
    // Problems are handed out through one global counter: a warp that needs k new problems takes the next k, so every
    // warp stays busy until the batch is exhausted.  (Measured: launch time = 4.45 ms + batch / 43.6 M/s.  The
    // constant is NOT load imbalance -- a static share per warp gave the same times -- but the drain of the trees that
    // are still open when the queue runs dry: a lane needs ~0.1 ms per node and the largest trees have > 100 nodes.)
    Solver sol;
    FlatCold<N> cold;
    sol.lane_ = lane;
    sol.P = &P;     // bound here, unconditionally: the compiler then reads the parameters from the constant bank
                    // instead of through a generic pointer (r01k ncu: LD.E of P->hull etc. on the SELECT path)
    bool have = false;
    int64_t i = 0;
    // Tail of the launch: when the queue has run dry, the lanes that are idle ADOPT open branches of the lanes of their
    // warp that are still searching (the launch time is 4.45 ms + batch / 43.6 M/s, and the 4.45 ms are exactly these
    // last, largest trees; see DESIGN 2.2).  The donor hands out untried regions of the shallowest open level of its
    // depth-first stack; an adopter sets the same problem up, follows the donor's region prefix without solving it and
    // searches that one branch from the donor's incumbent, keeping its best leaf in a scratch row; when it is done the
    // owner takes the better of the two.  Everything stays inside the warp: shuffles, no atomics, no global queue.
    const bool steal = STEAL && scratch != nullptr && P.max_nodes == 0;
    bool thief = false, drained = false;
    int owner = lane, pending = 0;
    double* const my_scratch = scratch ? scratch + ((size_t)blockIdx.x * 32 + lane) * N : nullptr;
    // A lane is either stepping its node QP (SELECT/STEP: the common, cheap trip) or waiting for node
    // work (store a finished problem, load the next one, NEXT + BUILD of a new node).  Node work is
    // several times the cost of a step and only ~1 lane in 6 needs it on a given trip, so the warp
    // lets waiting lanes accumulate and serves them together (r01d ncu: 7.7 of 32 lanes active when
    // every trip served them immediately).
    const int node_batch = P.node_batch;
    for (;;) {
        __syncwarp();
        const bool slow = !have || sol.state == Solver::S_DONE || sol.wants_node();
        const unsigned ms = __ballot_sync(0xffffffffu, slow);
        if (ms == 0xffffffffu || __popc(ms) >= node_batch) {
            if (STEAL && __builtin_expect(drained, 0)) {
                // adopters that finished their branch report to the owner of the problem
                unsigned rep = __ballot_sync(0xffffffffu, have && thief && sol.state == Solver::S_DONE && pending == 0);
                while (rep) {
                    const int r = __ffs(rep) - 1;
                    rep &= rep - 1;
                    const int o = __shfl_sync(0xffffffffu, owner, r);
                    const double v = __shfl_sync(0xffffffffu, sol.inc, r);
                    const unsigned long long bm = __shfl_sync(0xffffffffu, (unsigned long long)sol.best_modes, r);
                    const int nn = __shfl_sync(0xffffffffu, sol.nodes, r), ii = __shfl_sync(0xffffffffu, sol.iters, r);
                    // the owner's status is the worst of its own and its adopters' (time-out > node limit > numeric)
                    const int tr = __shfl_sync(0xffffffffu, (int)sol.trouble | ((int)sol.timeout << 1) | ((int)sol.limit << 2), r);
                    __syncwarp();
                    if (lane == o) {
                        --pending;
                        sol.nodes += nn; sol.iters += ii;
                        if (tr & 1) sol.trouble = true;
                        if (tr & 2) sol.timeout = true;
                        if (tr & 4) sol.limit = true;
                        if (v < sol.inc) {
                            sol.inc = v; sol.best_modes = bm;
                            const double* src = scratch + ((size_t)blockIdx.x * 32 + r) * N;
                            for (int j = 0; j < N; ++j) sol.best_[j] = src[j];
                        }
                    }
                    if (lane == r) { have = false; thief = false; owner = lane; }
                }
                __syncwarp();
            }
            if (have && !thief && sol.state == Solver::S_DONE && pending == 0) {
                const LocalResult R = sol.finish(u + (size_t)N * i, x + S * i, modes + (size_t)N * i);
                obj[i] = R.obj;
                status[i] = R.status;
                nodes[i] = R.nodes;
                if (qp_iters) qp_iters[i] = R.qp_iters;
                have = false;
            }
            // new work for idle lanes: a fresh problem from the queue, or (tail) a branch of a busy lane
            bool start = false, adopting = false;
            int a_l = 0, a_c = 0, a_owner = lane;
            unsigned long long a_modes = 0;
            long long a_t0 = 0;
            double a_inc = 0.0;
            const unsigned need = __ballot_sync(0xffffffffu, !have);
            if (need && !drained) {
                unsigned long long base = 0;
                if (lane == 0) base = atomicAdd(counter, (unsigned long long)__popc(need));
                base = __shfl_sync(0xffffffffu, base, 0);
                if (!have) {
                    const int64_t cand_i = (int64_t)base + __popc(need & ((1u << lane) - 1u));
                    if (cand_i < batch) { i = cand_i; start = true; }
                }
                if ((int64_t)base + __popc(need) > batch) drained = true;          // warp-uniform
            }
            if (STEAL && __builtin_expect(steal && drained, 0)) {
                // adopters pick up the owner's current incumbent
                const double oi = __shfl_sync(0xffffffffu, sol.inc, thief ? owner : lane);
                if (have && thief && oi < sol.inc) sol.inc = oi;
                unsigned idle = __ballot_sync(0xffffffffu, !have && !start);
                int l = -1, cb = 0, total = 0;
                const bool can = have && sol.state == Solver::S_NEXT && sol.open_level(l, cb, total) && total >= 2;   // adopters donate too
                unsigned don = __ballot_sync(0xffffffffu, can);
                for (int round = 0; round < 4 && don && idle; ++round) {
                    const int d = __ffs(don) - 1;
                    don &= don - 1;
                    const int dl = __shfl_sync(0xffffffffu, l, d), dcb = __shfl_sync(0xffffffffu, cb, d);
                    const int dtot = __shfl_sync(0xffffffffu, total, d);
                    const long long di = __shfl_sync(0xffffffffu, (long long)i, d);
                    const unsigned long long dm = __shfl_sync(0xffffffffu, (unsigned long long)sol.modes_pk, d);
                    const double dinc = __shfl_sync(0xffffffffu, sol.inc, d);
                    const long long dt0 = __shfl_sync(0xffffffffu, cold.t_start, d);     // the problem's clock
                    int m = __popc((unsigned)dcb) - (dtot == __popc((unsigned)dcb) ? 1 : 0);   // the donor keeps work
                    if (m > __popc(idle)) m = __popc(idle);
                    if (m <= 0) continue;
                    const bool me_idle = (idle >> lane) & 1u;
                    const int rk = __popc(idle & ((1u << lane) - 1u));
                    if (me_idle && rk < m) {
                        int bits = dcb;
                        for (int t = 0; t < rk; ++t) bits &= bits - 1;
                        a_c = __ffs(bits) - 1; a_l = dl; a_modes = dm; a_inc = dinc; a_owner = d; a_t0 = dt0;
                        i = di; start = true; adopting = true;
                    }
                    if (lane == d) {
                        int bits = dcb, rm = 0;
                        for (int t = 0; t < m; ++t) { rm |= bits & -bits; bits &= bits - 1; }
                        sol.set_cand(dl, dcb & ~rm);
                        pending += m;
                    }
                    idle = __ballot_sync(0xffffffffu, !have && !start);
                }
            }
            if (start) {
                sol.setup(smem + lane, &P, flags[i], mass[i], x0 + 2 * i, xf ? xf + S * i : nullptr,
                          xb ? xb + S * i : nullptr, xl ? xl + S * i : nullptr,
                          adopting ? my_scratch : x + S * i + (N + 2), &cold);
                if (STEAL && adopting) {
                    sol.adopt_prefix(a_modes, a_l, a_c, a_inc);
                    cold.t_start = a_t0;       // one problem, one budget: an adopted branch keeps the owner's clock
                }
                else if (HINTS && P.hint) sol.apply_hint(P.hint + (size_t)N * i);
                have = true; thief = adopting; owner = a_owner;
            }
            if (!__any_sync(0xffffffffu, have)) break;
            if (have) sol.trip_node();
        }
        if (have) sol.trip_step();
    }
}

static int env_int(const char* name, int dflt) {
    const char* e = getenv(name);
    return e ? atoi(e) : dflt;
}

template <int N>
static cudaError_t launch_flat(const LocalParams& P, unsigned long long* counter, double* steal_scratch, int64_t batch, const int32_t* flags, const double* mass,
                               const double* x0, const double* xf, const double* xb, const double* xl, double* u,
                               double* x, int32_t* modes, double* obj, int32_t* status, int32_t* nodes,
                               int32_t* qp_iters, cudaStream_t stream) {
    const size_t smem = (size_t)FlatLayout<N>::SIZE * 32 * sizeof(double);
    // attributes and occupancy are per DEVICE (several devices per process: Context(device)): cached per device
    int dev = 0;
    cudaGetDevice(&dev);
    static int grid_cache[HVP_MAX_DEVICES] = {0};
    int uncached = 0;
    int& grid_full = (dev >= 0 && dev < HVP_MAX_DEVICES) ? grid_cache[dev] : uncached;
    if (!grid_full) {
        cudaError_t e = cudaSuccess;
        const void* fns[3] = {(const void*)flat_miqp_kernel<N, true, false>, (const void*)flat_miqp_kernel<N, false, false>,
                              (const void*)flat_miqp_kernel<N, true, true>};
        for (int v = 0; v < 3; ++v) {
            const void* fn = fns[v];
            e = cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
            if (e != cudaSuccess) return e;
            e = cudaFuncSetAttribute(fn, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared);
            if (e != cudaSuccess) return e;
        }
        int sms = 0, per_sm = 0;
        cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, flat_miqp_kernel<N, true, false>, 32, smem);
        if (e != cudaSuccess) return e;
        grid_full = sms * (per_sm > 0 ? per_sm : 1);
    }
    // persistent grid: every resident warp slot, but never more warps than 32-problem shares
    int64_t g = (batch + 31) / 32;
    static const int gdiv = env_int("HVP_FLAT_GRID_DIV", 1);
    if (g > grid_full / gdiv) g = grid_full / gdiv;
    LocalParams Q = P;
    static const int nb = env_int("HVP_NODE_BATCH", 0), dv = env_int("HVP_FLAT_DIVE", -1);
    if (nb > 0) Q.node_batch = nb;
    if (dv >= 0) Q.dive = dv;
    static const int steal_on = env_int("HVP_FLAT_STEAL", 1);
    if ((size_t)g * 32 * N > HVP_STEAL_SLOT_DOUBLES) steal_scratch = nullptr;
    cudaError_t e = cudaMemsetAsync(counter, 0, sizeof(unsigned long long), stream);
    if (e != cudaSuccess) return e;
    if (Q.hint)              // MIP start given: the instantiation with the hint entry (adoption on when the scratch allows)
        flat_miqp_kernel<N, true, true><<<(unsigned)g, 32, smem, stream>>>(Q, batch, flags, mass, x0, xf, xb, xl, u, x, modes, obj,
                                                                          status, nodes, qp_iters, counter,
                                                                          steal_on ? steal_scratch : nullptr);
    else if (steal_on && steal_scratch)
        flat_miqp_kernel<N, true, false><<<(unsigned)g, 32, smem, stream>>>(Q, batch, flags, mass, x0, xf, xb, xl, u, x, modes, obj,
                                                                           status, nodes, qp_iters, counter, steal_scratch);
    else
        flat_miqp_kernel<N, false, false><<<(unsigned)g, 32, smem, stream>>>(Q, batch, flags, mass, x0, xf, xb, xl, u, x, modes, obj,
                                                                            status, nodes, qp_iters, counter, nullptr);
    return cudaGetLastError();
}

// 0 auto, 2 coop, 3 flat
static int kernel_choice() {
    static int v = -1;
    if (v < 0) {
        const char* e = getenv("HVP_LOCAL_KERNEL");
        v = 0;
        if (e && strcmp(e, "coop") == 0) v = 2;
        if (e && strcmp(e, "flat") == 0) v = 3;
    }
    return v;
}

cudaError_t launch_local_miqp(const LocalParams& P, unsigned long long* counter, double* steal_scratch, int64_t batch, const int32_t* flags, const double* mass,
                              const double* x0, const double* xf, const double* xb, const double* xl,
                              double* u, double* x, int32_t* modes, double* obj, int32_t* status,
                              int32_t* nodes, int32_t* qp_iters, cudaStream_t stream) {
    if (batch <= 0) return cudaSuccess;
    // throughput path: persistent flat kernel (one problem per lane) once the batch fills the
    // machine; latency path: cooperative kernel (8 lanes per problem) for small batches
    const int choice = kernel_choice();
    const bool flat_ok = P.N >= 4 && P.N <= 9;
    if (flat_ok && (choice == 3 || (choice == 0 && batch >= FLAT_MIN_BATCH))) {
#define HVP_FLAT(NN) case NN: return launch_flat<NN>(P, counter, steal_scratch, batch, flags, mass, x0, xf, xb, xl, u, x, modes, obj, status, nodes, qp_iters, stream);
        switch (P.N) { HVP_FLAT(4) HVP_FLAT(5) HVP_FLAT(6) HVP_FLAT(7) HVP_FLAT(8) HVP_FLAT(9) default: break; }
#undef HVP_FLAT
    }
    {
        // a handful of trees (one scenario-timestep = n MIQPs): several workers per tree
        static const int splitM = env_int("HVP_COOP_SPLIT_M", 8);
        if (P.N <= 8 && batch <= COOP_SPLIT_MAX && splitM > 1 && splitM <= 32 && steal_scratch && P.max_nodes == 0 &&
            2 * P.N + 2 * (P.N + 1) + 4 <= COOP_SPLIT_ROW) {
            const size_t head = (size_t)COOP_SPLIT_MAX * (sizeof(unsigned) + sizeof(unsigned long long));
            unsigned* done = reinterpret_cast<unsigned*>(steal_scratch);
            unsigned long long* keys = reinterpret_cast<unsigned long long*>(reinterpret_cast<char*>(steal_scratch) + COOP_SPLIT_MAX * sizeof(unsigned));
            double* rows = reinterpret_cast<double*>(reinterpret_cast<char*>(steal_scratch) + head);
            cudaError_t e = cudaMemsetAsync(steal_scratch, 0xFF, head, stream);
            if (e != cudaSuccess) return e;
            coop_split_kernel<8><<<(unsigned)(batch * splitM), 32, 0, stream>>>(P, batch, splitM, flags, mass, x0, xf, xb, xl, u, x,
                                                                                modes, obj, status, nodes, qp_iters, done, keys, rows);
            return cudaGetLastError();
        }
        if (P.N <= 8) {
            if (batch <= COOP_SPREAD_MAX) {
                coop_miqp_kernel<8><<<(unsigned)batch, 32, 0, stream>>>(P, batch, flags, mass, x0, xf, xb, xl, u, x, modes,
                                                                      obj, status, nodes, qp_iters, 1);
                return cudaGetLastError();
            }
            const int per_block = COOP_BLOCK / 8;
            const unsigned g = (unsigned)((batch + per_block - 1) / per_block);
            coop_miqp_kernel<8><<<g, COOP_BLOCK, 0, stream>>>(P, batch, flags, mass, x0, xf, xb, xl, u, x, modes, obj,
                                                             status, nodes, qp_iters, 0);
        } else {
            if (batch <= COOP_SPREAD_MAX) {
                coop_miqp_kernel<16><<<(unsigned)batch, 32, 0, stream>>>(P, batch, flags, mass, x0, xf, xb, xl, u, x, modes,
                                                                       obj, status, nodes, qp_iters, 1);
                return cudaGetLastError();
            }
            const int per_block = COOP_BLOCK / 16;
            const unsigned g = (unsigned)((batch + per_block - 1) / per_block);
            coop_miqp_kernel<16><<<g, COOP_BLOCK, 0, stream>>>(P, batch, flags, mass, x0, xf, xb, xl, u, x, modes, obj,
                                                              status, nodes, qp_iters, 0);
        }
        return cudaGetLastError();
    }
    return cudaErrorInvalidConfiguration;
}

}  // namespace hvp
