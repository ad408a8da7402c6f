/*
 * hvp.h -- C ABI of the B200-native hybrid-MPC hot path (libhvp.so).
 *
 * This is the drop-in boundary for ONE path of Kevindqz/hybrid-vehicle-platoon: the
 * per-timestep MLD/PWA mixed-integer QP solves and the nonlinear hybrid rollout + stage cost.
 * The reference has no FFI for this path (it is Python calling gurobipy); the entry points
 * below are what its Python layer binds through ctypes (INTEGRATION.md shows the stubs).
 * `file:line` citations are into the reference tree.
 *
 * Conventions
 *   - extern "C", plain pointers and sizes, no torch / CUDA types in signatures
 *     (`stream` is a cudaStream_t passed as void*; NULL = the context's own stream; pass
 *     cudaStreamLegacy ((void*)1) for the legacy default stream).
 *   - `*_dev` entry points take DEVICE pointers owned by the caller (e.g. torch tensors'
 *     data_ptr()); they enqueue work on `stream` and return without synchronising.
 *   - `*_host` entry points take HOST pointers, copy host->device, run the same kernels, copy the
 *     results back and synchronise before returning (the reference-facing call: numpy in, numpy out).
 *   - All arrays are dense row-major, float64 unless stated.  Batches are [batch][...].
 *   - Every function returns 0 on success, <0 on API misuse / CUDA error (text via
 *     hvp_last_error).  Per-problem outcomes are reported in status[] with the Gurobi codes the
 *     reference tests for (mpcs/mpc_gear.py:119,156; fleet_event_based.py:323):
 *     2 OPTIMAL, 3 INFEASIBLE, 8 NODE_LIMIT, 12 NUMERIC.
 *   - A context is bound to one device and one stream and is not thread-safe; distinct contexts
 *     are independent.  There is NO CPU fallback: without a CUDA device every call fails.
 */
#ifndef HVP_H
#define HVP_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define HVP_VERSION 101

/* status[] codes (Gurobi numbering, mpcs/mpc_gear.py:119) */
#define HVP_OPTIMAL 2
#define HVP_INFEASIBLE 3
#define HVP_NODE_LIMIT 8
#define HVP_TIME_LIMIT 9 /* time_limit_ms ran out: the best solution found so far is returned (Gurobi TIME_LIMIT) */
#define HVP_NUMERIC 12

/* per-vehicle role flags of a local problem (fleet_decent_mld.py:33-45: is_front/is_leader/is_trailer) */
#define HVP_FRONT 1
#define HVP_LEADER 2
#define HVP_TRAILER 4

/* rollout err[] codes = code | vehicle<<8 | substep<<16 of the FIRST exception the reference
 * would raise (models.py:32-42,119-122); 0 = none */
#define HVP_ERR_VELOCITY_BOUNDS 1 /* models.py:119-122 / :34-35 */
#define HVP_ERR_GEAR_INDEX 2      /* models.py:32-33 */
#define HVP_ERR_GEAR_RANGE 3      /* models.py:39-42 */

int hvp_version(void);
/* copies the calling thread's last error text into buf (NUL-terminated); returns its length */
int hvp_last_error(char* buf, int len);
/* number of visible CUDA devices (<=0: none -> nothing in this library can run) */
int hvp_device_count(void);

/* ---- context ------------------------------------------------------------------------------ */
typedef struct hvp_ctx hvp_ctx;
int hvp_ctx_create(int device, hvp_ctx** out);
int hvp_ctx_destroy(hvp_ctx* ctx);
/* the context's own stream as a cudaStream_t (for callers that want to order work after it) */
void* hvp_ctx_stream(hvp_ctx* ctx);
int hvp_ctx_synchronize(hvp_ctx* ctx);
/* number of kernels this context has launched so far (bench.py's gpu_launches) */
int64_t hvp_ctx_launch_count(hvp_ctx* ctx);
/* duration in ms of the kernels of the most recent *_host/_dev call made through the context's
 * timed wrappers (CUDA events on the context stream); <0 if none */
float hvp_ctx_last_kernel_ms(hvp_ctx* ctx);

/* ---- (c) rollout + stage cost: replaces PlatoonEnv.step (env.py:182-212) -------------------
 * = get_stage_cost on the PRE-step state (env.py:126-180), optional gear derivation
 * (env.py:198-204 -> models.py:494-515) and Platoon.step_platoon (models.py:236-257: ten explicit
 * Euler sub-steps of Vehicle.step models.py:114-125 with GearTransimission.get_traction :30-51). */
typedef struct {
    int32_t n;            /* vehicles per platoon */
    int32_t leader_index; /* env.py:31 */
    int32_t flags;        /* HVP_ENV_* */
    int32_t reserved;
    double d0, t0;        /* spacing policy sigma(x) = [-t0*v - d0, 0] (misc/spacing_policy.py:13-37) */
    double d_safe;        /* env.py:38 */
} hvp_env_desc;
#define HVP_ENV_QUADRATIC 1         /* env.py:55-58: x'Qx, else ||Qx||_1 */
#define HVP_ENV_REAL_VEHICLE_REF 2  /* env.py:141-151 */
#define HVP_ENV_MASS_PER_SCENARIO 4 /* mass is [batch][n] instead of [n] */

/* x [batch][2n] = [p0 v0 p1 v1 ...] (env.py:79 ordering), u [batch][n], gear [batch][n] int32 or
 * NULL (derive from velocity), mass [n] / [batch][n] / NULL (800 kg), leader [batch][2] =
 * leader_x[:, step_counter].  Outputs: x_out [batch][2n], cost [batch], viol [batch] (0/1,
 * env.py:165-176), err [batch].  x_out of a scenario with err != 0 is NaN. */
int hvp_rollout_step_dev(hvp_ctx* ctx, const hvp_env_desc* desc, int64_t batch, const double* x,
                         const double* u, const int32_t* gear, const double* mass,
                         const double* leader, double* x_out, double* cost, uint8_t* viol,
                         int32_t* err, void* stream);
int hvp_rollout_step_host(hvp_ctx* ctx, const hvp_env_desc* desc, int64_t batch, const double* x,
                          const double* u, const int32_t* gear, const double* mass,
                          const double* leader, double* x_out, double* cost, uint8_t* viol,
                          int32_t* err);

/* ---- (a) per-vehicle local MIQP: replaces LocalMpcMld(...).solve_mpc(state) ----------------
 * Problem definition: fleet_decent_mld.py:61-208 (identical in fleet_seq_mld.py:63-219) on top
 * of dmpcpwa MpcMld (PWA->MLD, SURVEY.md 8a rows A1/A2/A7), pwa_gear model (models.py:397-492).
 * Solved to proven optimality (gap 0) by branch-and-bound over the PWA region sequence. */
typedef struct {
    int32_t N;          /* horizon (<= 12) */
    int32_t max_nodes;  /* per problem; 0 = unlimited */
    double d0, t0;      /* spacing policy */
    double tight;       /* accel_cnstr_tightening (fleet_decent_mld.py:43) */
    /* Solver options (SURVEY.md 8b; Gurobi parameters of mpcs/mpc_gear.py:182-186, Q12).  mip_gap: relative gap at
     * which a node is pruned (Gurobi MIPGap, default there 1e-4); 0 = proven optimal.  time_limit_ms: budget per
     * problem, measured on the device from the moment the problem is picked up; when it runs out the incumbent is
     * returned with status HVP_TIME_LIMIT (9); 0 = none.  Sub-trees that other lanes or warps search for the problem
     * (the split of small batches, adoption in the tail of a flat launch) run on the same budget, and a time-out in
     * any of them makes the problem's status HVP_TIME_LIMIT. */
    double mip_gap;
    double time_limit_ms;
    /* Optional incumbent hint for hvp_local_miqp_dev: DEVICE pointer to [batch][N] int32 region sequences (the codes
     * modes[] returns) to be tried first -- in a closed loop the previous step's optimal sequence shifted by one
     * stage (fleet_decent_mld.py:314-316 calls solve_mpc once per timestep with a warm model; Gurobi does the same
     * with its MIP start).  Advice only: the result is the proven optimum with or without it.  NULL = none; ignored
     * by the *_host entry point and by batches small enough for the cooperative kernel. */
    const int32_t* modes_hint;
} hvp_local_desc;

/* flags [batch] (HVP_FRONT|HVP_LEADER|HVP_TRAILER), mass [batch], x0 [batch][2],
 * xf / xb / xl [batch][2][N+1] = x_front / x_back / leader_x parameters (set_x_front, set_x_back,
 * set_leader_x: fleet_decent_mld.py:210-223); unused ones may be NULL.
 * Outputs: u [batch][N], x [batch][2][N+1], modes [batch][N] int32 (active PWA region per stage,
 * = argmax_r delta[r,k]), obj [batch] (objVal incl. constant terms; +inf if infeasible),
 * status [batch] int32, nodes [batch] int32 (B&B nodes = QPs solved), qp_iters [batch] int32 or
 * NULL (active-set iterations summed over the nodes). */
int hvp_local_miqp_dev(hvp_ctx* ctx, const hvp_local_desc* desc, int64_t batch, const int32_t* flags,
                       const double* mass, const double* x0, const double* xf, const double* xb,
                       const double* xl, double* u, double* x, int32_t* modes, double* obj,
                       int32_t* status, int32_t* nodes, int32_t* qp_iters, void* stream);
int hvp_local_miqp_host(hvp_ctx* ctx, const hvp_local_desc* desc, int64_t batch, const int32_t* flags,
                        const double* mass, const double* x0, const double* xf, const double* xb,
                        const double* xl, double* u, double* x, int32_t* modes, double* obj,
                        int32_t* status, int32_t* nodes, int32_t* qp_iters);

/* ---- (a) compiled MPC formulations: centralized, event-based, ADMM, discrete gears --------------
 * One handle = one MPC model, built once (the reference builds its Gurobi model once per controller)
 * and solved for batches of (initial state, parameters).  Replaces
 *   HVP_MPC_CENT   MpcMldCent(...).solve_mpc            mpcs/cent_mld.py:9-182      (+ set_leader_traj)
 *   HVP_MPC_LOCAL  LocalMpcMld / LocalMpcGear            fleet_decent_mld.py:21-253, fleet_seq_mld.py:21-264
 *   HVP_MPC_EVENT  event-based LocalMpc / LocalMpcGear   fleet_event_based.py:26-376  (solve_mpc)
 *   HVP_MPC_ADMM   LocalMpcADMM / LocalMpcGear           fleet_naive_admm.py:24-290
 *   HVP_MPC_GADMM  fixed-sequence LocalMpc(MpcSwitching) fleet_g_admm.py:22-205       (pass fixed_modes)
 * on model HVP_MODEL_PWA_GEAR (7 PWA regions, models.py:397-492) or HVP_MODEL_FRICTION_GEAR (2 friction
 * regions x 6 discrete gears = MpcGear.setup_gears on pwa_friction, mpcs/mpc_gear.py:30-114,
 * models.py:288-332; the penalised/limited input is the throttle u_g).
 *
 * Parameter vector of one problem, params[npar]: blocks of (2, N+1) row-major [p_0..p_N, v_0..v_N]:
 *   CENT : leader_traj
 *   LOCAL: x_front, x_back, leader_x                     (set_x_front / set_x_back / set_leader_x)
 *   EVENT: leader_x, x_f2, x_b2                          (set_leader_x / set_x_f2 / set_x_b2)
 *   ADMM : leader_x, y_front, z_front, y_back, z_back    (set_leader_x / set_front_vars / set_back_vars)
 *   GADMM: x_ref, then y and z, each (2 (1 + n_front + n_behind), N+1) in augmented order
 *          [copies in front..., own state, copies behind...]
 * Unused blocks must still be present (any finite values).  Extra decision variables returned in
 * extra[n_extra]: ADMM [x_front if not FRONT][x_back if not TRAILER]; GADMM the neighbour copies in
 * augmented order; others none.
 * Local vehicles are ordered front to back: x0 [batch][n_local][2], mass [batch][n_local]. */
#define HVP_MPC_CENT 1
#define HVP_MPC_LOCAL 2
#define HVP_MPC_EVENT 3
#define HVP_MPC_ADMM 4
#define HVP_MPC_GADMM 5
#define HVP_MODEL_PWA_GEAR 0
#define HVP_MODEL_FRICTION_GEAR 1
#define HVP_REAL_VEHICLE_REF 8 /* flags bit: real_vehicle_as_reference (cent_mld.py:31, fleet_seq_mld.py:211-219) */
#define HVP_NO_LEADER (-100)   /* EVENT: rel_leader_index = None */
typedef struct {
    int32_t kind;         /* HVP_MPC_* */
    int32_t model;        /* HVP_MODEL_* */
    int32_t n_local;      /* vehicles whose inputs are decided (CENT: n; EVENT: 2-3; others: 1) */
    int32_t N;            /* horizon */
    int32_t flags;        /* HVP_FRONT|HVP_LEADER|HVP_TRAILER (LOCAL, ADMM, GADMM: HVP_LEADER) | HVP_REAL_VEHICLE_REF */
    int32_t leader_index; /* CENT: leader_index; EVENT: rel_leader_index in {-1,0,1} or HVP_NO_LEADER */
    int32_t n_front;      /* EVENT: num_vehicles_in_front (0..2); GADMM: copies in front of own state */
    int32_t n_behind;     /* EVENT: num_vehicles_behind (0..2);   GADMM: copies behind own state */
    int32_t max_nodes;    /* per problem; 0 = unlimited */
    int32_t one_norm;     /* 0: 2-norm cost (MIQP); 1: 1-norm cost sum |Q e| (MILP; quadratic_cost=False, cent_mld.py:58-61) */
    double d0, t0;        /* spacing policy */
    double tight;         /* accel_cnstr_tightening */
    double rho;           /* ADMM / GADMM penalty */
    double mip_gap;       /* as in hvp_local_desc; 0 = proven optimal */
    double time_limit_ms; /* as in hvp_local_desc; 0 = none */
} hvp_mpc_desc;
typedef struct hvp_mpc hvp_mpc;
int hvp_mpc_create(hvp_ctx* ctx, const hvp_mpc_desc* desc, hvp_mpc** out);
int hvp_mpc_destroy(hvp_mpc* mpc);
/* info[8] = { n_var (variables of a node QP after the compile-time elimination of free copies that appear in no
 * row), n_extra (free copies REPORTED in `extra`), n_param, n_modes, n_local, N, n_rows (coupling), smem bytes per warp } */
int hvp_mpc_info(const hvp_mpc* mpc, int32_t* info);
/* PWA mode table of the model: lo/hi velocity interval and the gear (1..6) of each of n_modes modes */
int hvp_mpc_mode_table(const hvp_mpc* mpc, double* lo, double* hi, int32_t* gear);
/* x0 [batch][n_local][2], mass [batch][n_local], params [batch][n_param], fixed_modes [batch][n_local][N]
 * int32 or NULL (NULL: branch and bound over the modes; given: the single fixed-mode QP).
 * Outputs: u [batch][n_local][N], x [batch][n_local][2][N+1], extra [batch][n_extra] or NULL,
 * modes [batch][n_local][N] int32, obj, status, nodes [batch], qp_iters [batch] or NULL. */
int hvp_mpc_solve_dev(hvp_mpc* mpc, int64_t batch, const double* x0, const double* mass, const double* params,
                      const int32_t* fixed_modes, double* u, double* x, double* extra, int32_t* modes,
                      double* obj, int32_t* status, int32_t* nodes, int32_t* qp_iters, void* stream);
int hvp_mpc_solve_host(hvp_mpc* mpc, int64_t batch, const double* x0, const double* mass, const double* params,
                       const int32_t* fixed_modes, double* u, double* x, double* extra, int32_t* modes,
                       double* obj, int32_t* status, int32_t* nodes, int32_t* qp_iters);

/* Multi-GPU split of LARGE trees (north_star: "allreduce-min the incumbent objective bound when a single large
 * MIQP's tree is split across GPUs"; the reference has no counterpart -- Gurobi's threads play this role,
 * mpcs/mpc_gear.py:185-186).  Every device of `world` calls this with the SAME batch; device `rank` searches, for
 * every problem, the sub-trees whose depth-`prefix_depth` mode-prefix ordinal o has o % world == rank (dealt to the
 * `groups` warps this device gives each problem by (o / world) % groups; the warps of a device share their
 * incumbent through global memory).  incumbent [batch] (device, or NULL = +inf) seeds the bound: only leaves
 * strictly better are accepted.  node_budget > 0 stops every warp after that many nodes (every node counts: solved,
 * pruned, infeasible, leaf; status 8) -- the cheap first wave that produces a bound to exchange; 0 searches the share to
 * completion, and then warps of this device that run out of work adopt sub-trees of busy ones (any problem of the batch).  obj [batch] = best leaf of
 * THIS device's share (+inf: none better than the incumbent; status 3).  The caller combines the devices with
 * allreduce(min) over obj (NCCL) and takes u/x/modes from the device that attains it
 * (hybrid_vehicle_platoon_b200/dist.py: solve_tree_split).  prefix_depth 0 = the handle's default. */
int hvp_mpc_solve_shard_dev(hvp_mpc* mpc, int64_t batch, const double* x0, const double* mass, const double* params,
                            int32_t rank, int32_t world, int32_t groups, int32_t prefix_depth, int32_t node_budget,
                            const double* incumbent, double* u, double* x, double* extra, int32_t* modes, double* obj,
                            int32_t* status, int32_t* nodes, int32_t* qp_iters, void* stream);

/* eval_cost of the event-based LocalMpc (fleet_event_based.py:308-327): cost of a guess with x[:, :N]
 * and u pinned -- xg [batch][n_local][2][N+1] (column N is ignored: the last state is free),
 * ug [batch][n_local][N]; the initial condition is xg[..., 0].  cost [batch] = objVal, +inf if the guess
 * is infeasible for the MLD model (tolerance 1e-6 = Gurobi's FeasibilityTol). */
int hvp_mpc_eval_dev(hvp_mpc* mpc, int64_t batch, const double* mass, const double* params, const double* xg,
                     const double* ug, double* cost, void* stream);
int hvp_mpc_eval_host(hvp_mpc* mpc, int64_t batch, const double* mass, const double* params, const double* xg,
                      const double* ug, double* cost);

/* ---- measurement helpers (bench.py) ---------------------------------------------------------
 * FP64 FMA issue peak of the device: `iters` dependent-chain FMAs x 8 independent chains per
 * thread over a full grid; returns achieved TFLOP/s (2 flop per FMA) in *tflops. */
int hvp_microbench_fp64(hvp_ctx* ctx, int iters, double* tflops);
/* measured shared-memory read bandwidth of the whole device in GB/s (SURVEY 8d: smem roofline of the QP kernels) */
int hvp_microbench_smem(hvp_ctx* ctx, int iters, double* gbs);

/* ---- fused coordinator glue of the switching ("g") ADMM controller ---------------------------------
 * Replaces, per consensus round and for all scenarios at once, what fleet_g_admm.py:255-301 and the round logic of
 * dmpcpwa's GAdmmCoordinator do between two batches of local QPs: z-update (mean of the copies of each vehicle's
 * trajectory), y-update, adoption of the solved QPs' inputs, PWA roll-out of the inputs and re-identification of the
 * region sequences (the next round's fixed_modes), and the packing of the next round's parameter vectors.
 * Roles: [0] vehicle 0 (GADMM, leader, n_behind = 1), [1] vehicle n-1 (n_front = 1, n_behind = 0), [2] vehicles
 * 1..n-2 (n_front = n_behind = 1; unused when n == 2).  A role's buffers are the arguments of ITS hvp_mpc_solve_dev
 * call, problems ordered [scenario][vehicle of the role]: params / x0 / mass / fixed_modes are WRITTEN here (the next
 * solve's inputs), u / x / extra / obj / status are READ (the last solve's outputs; not with init = 1).
 * init = 1 starts a warm start: y = 0, z = the roll-out of `u`, ok = 1.  All pointers are device pointers. */
typedef struct {
    double* params; double* x0; double* mass; int32_t* fixed_modes;
    const double* u; const double* x; const double* extra; const double* obj; const int32_t* status;
} hvp_gadmm_role;
typedef struct {
    int32_t n, N, S, init;
    double rho;
    double mug, edge[6], cf[7], bg[7], dd[7]; /* pwa_gear regions: v+ = (1 - cf/m) v + (bg/m) u - mug - dd/m, edges between them */
    hvp_gadmm_role role[3];
    const double* x;    /* [S][n][2]      */
    const double* mass; /* [S][n]         */
    const double* lwin; /* [S][2][N+1]    leader trajectory window of this timestep */
    double* y;          /* [S][n][3][2][N+1]  multipliers: front copy, own, back copy */
    double* u;          /* [S][n][N]      inputs: start / previous round in, updated out */
    double* tr;         /* [S][n][2][N+1] PWA roll-out of u (out) */
    double* cost;       /* [S]            sum of the solved QPs' objectives (out) */
    uint8_t* ok;        /* [S]            1 while every QP of every round was solved */
} hvp_gadmm_round;
int hvp_gadmm_round_dev(hvp_ctx* ctx, const hvp_gadmm_round* g, void* stream);

/* ---- fused observe step of the decentralized / sequential controllers -----------------------------------
 * fleet_decent_mld.py:329-331, :421-428 for all scenarios at once: every vehicle's constant-velocity extrapolation
 * (p_{k+1} = p_k + ts v_k, summed sequentially as the reference does) is written as x_front of the vehicle behind it
 * and x_back of the vehicle in front, and the leader gets leader_x[:, t : t + N + 1].  t is read from DEVICE memory
 * so that a timestep can be replayed as a CUDA graph. */
typedef struct {
    int32_t n, N, S, leader_index;
    int64_t leader_len;           /* columns of the leader trajectory */
    int32_t leader_per_scenario;  /* leader_x is [S][2][leader_len] (1) or [2][leader_len] shared (0) */
    int32_t reserved;
    double ts;
    const double* x;              /* [S][n][2] */
    const double* leader_x;
    const int64_t* t;             /* device pointer: timestep index */
    double* xf; double* xb; double* xl; /* [S][n][2][N+1] each; rows without a neighbour / not the leader are left alone */
} hvp_decent_observe;
int hvp_decent_observe_dev(hvp_ctx* ctx, const hvp_decent_observe* g, void* stream);

/* ---- fused z- / y-update of a naive-ADMM consensus round ------------------------------------------------
 * fleet_naive_admm.py:421-468 for all scenarios at once, read straight from the outputs of the role solves
 * (hvp_mpc_solve_dev of the ADMM formulations: x = own prediction, extra = the copies x_front / x_back), writing the
 * consensus variables and the next round's parameter vectors [leader window | y_front | z_front | y_back | z_back].
 * role_of[i] = index into role[] of vehicle i; problems of a role are ordered [scenario][vehicle of the role]. */
typedef struct {
    double* params; const double* x; const double* extra;
    int32_t has_front, has_back;  /* the role's formulation holds an x_front / x_back copy (not FRONT / not TRAILER) */
} hvp_admm_role;
typedef struct {
    int32_t n, N, S, nroles;
    int32_t pack_only;            /* 1: only (re)write the parameter vectors from the consensus variables (start of a timestep) */
    int32_t reserved;
    double rho;
    hvp_admm_role role[4];
    int32_t role_of[64];
    const double* lwin;           /* [S][2][N+1] leader window (a parameter block of every role) */
    double* y_front; double* y_back; double* zf; double* zb; double* xs; /* [S][n][2][N+1] each */
} hvp_admm_round;
int hvp_admm_round_dev(hvp_ctx* ctx, const hvp_admm_round* g, void* stream);

/* ---- fused glue of a naive-ADMM timestep ----------------------------------------------------------------------
 * What ADMMCoordinator.get_control / on_timestep_end (fleet_naive_admm.py:379-587) do around the role solves, for all
 * S scenarios at once, one thread per (scenario, vehicle); the z / y update is the device code of hvp_admm_round_dev.
 * role_of[i] = index into role[] of vehicle i; the problems of a role (the rows of its hvp_mpc_solve_dev call) are
 * ordered [scenario][vehicle of the role].  t and the round index r are read from DEVICE memory (the caller advances
 * them) so that a round can be replayed as a CUDA graph.  A vehicle whose solve is not optimal (status != 2)
 * contributes zeros for its own prediction and its copies and gets u0 = 0 and gear 6, as solve_mpc(raises=False)
 * gives it (LocalMpcADMM._post).  Three phases:
 *   HVP_ADMM_PACK  (start of a timestep, before round 0): the role rows x0 = x[s][i]; when t > 0 the shifted previous
 *       predictions zf[i] = xs[i-1], zb[i] = xs[i+1] with column 0 dropped and the last one repeated (no re-extrapolated
 *       position: get_predicted_state(shifted=True)); then the parameter rows [lwin | y_front | zf | y_back | zb],
 *       lwin = leader_x[:, t : t+N+1] (a column past the end of leader_x reads its last column).
 *   HVP_ADMM_ROUND (after the role solves of round r): xs, zf, zb, y_front, y_back and the parameter rows exactly as
 *       hvp_admm_round_dev (same order of additions, a true division by 3), lwin as in PACK;
 *       ND[t][s] = max(ND[t][s], nodes of every vehicle); failed_at[s] = (t, r, status) of the first solve of the
 *       episode that was not optimal -- the lowest vehicle index within the first such round -- (-1, -1, 0): none;
 *       the row is reset at t == 0, r == 0.
 *   HVP_ADMM_ADOPT (after the last round, before the rollout): u0 = u[..., 0], with a gear output gear0 =
 *       mode_gear[modes[..., 0]] (mode index clamped to [0, n_modes)); U_log[t] = u0, followed by the gears as doubles
 *       when gear0 is given (w = 2n: the reference's [u_g ; gears]; else w = n); ST[t] = the last round's statuses.
 * ND, failed_at, U_log and ST are written only for 0 <= t < T.  All pointers are device pointers. */
#define HVP_ADMM_PACK 0
#define HVP_ADMM_ROUND 1
#define HVP_ADMM_ADOPT 2
typedef struct {
    double* params;               /* PACK / ROUND out: [rows][5 * 2(N+1)] */
    double* x0;                   /* PACK out: [rows][1][2] */
    const double* u; const double* x; const double* extra; const int32_t* modes; const int32_t* status;
    const int32_t* nodes;         /* solve outputs: [rows][N], [rows][2][N+1], [rows][ne], [rows][N], [rows], [rows] */
    int32_t has_front, has_back;  /* the role's formulation holds an x_front / x_back copy (not FRONT / not TRAILER) */
} hvp_admm_step_role;
typedef struct {
    int32_t n, N, S, phase;       /* phase: HVP_ADMM_PACK | HVP_ADMM_ROUND | HVP_ADMM_ADOPT */
    int32_t nroles;               /* 1..4 */
    int32_t leader_per_scenario;  /* leader_x is [S][2][leader_len] (1) or [2][leader_len] shared (0) */
    int64_t leader_len;           /* PACK / ROUND: columns of the leader trajectory (>= 1) */
    int64_t T;                    /* ROUND / ADOPT: rows of the episode logs */
    double rho;
    int32_t n_modes;              /* ADOPT with gear0: entries of mode_gear (1..16) */
    int32_t reserved;
    int32_t mode_gear[16];
    hvp_admm_step_role role[4];
    int32_t role_of[64];
    const int64_t* t;             /* device pointer: timestep index */
    const int32_t* r;             /* device pointer: round index within the timestep (ROUND) */
    const double* x;              /* PACK: [S][n][2] */
    const double* leader_x;       /* PACK / ROUND */
    double* y_front; double* y_back; double* zf; double* zb; double* xs; /* [S][n][2][N+1] each */
    int32_t* ND;                  /* ROUND: [T][S] */
    int32_t* failed_at;           /* ROUND: [S][3] */
    double* u0; int32_t* gear0;   /* ADOPT out: [S][n] each; gear0 NULL: no gears */
    double* U_log; int32_t* ST;   /* ADOPT: [T][S][w], [T][S][n] */
} hvp_admm_step;
int hvp_admm_step_dev(hvp_ctx* ctx, const hvp_admm_step* g, void* stream);

/* ---- fused glue of a centralized timestep ---------------------------------------------------------------------
 * What TrackingCentralizedAgent (fleet_cent_mld.py:22-32) and MpcMldCent / MpcGearCent.solve_mpc (mpcs/mpc_gear.py:
 * 116-135) do around the solve, for all S scenarios at once, one thread per (scenario, vehicle).  t is read from DEVICE
 * memory so that a timestep can be replayed as a CUDA graph.  Two phases:
 *   HVP_CENT_PACK  (before hvp_mpc_solve_dev of the CENT handle): params[s][0 : 2(N+1)] = leader_x[:, t : t+N+1], the
 *       CENT parameter block 0 ([p_t..p_t+N, v_t..v_t+N]); the rest of each params row is left alone.  leader_x is
 *       [2][leader_len] shared or [S][2][leader_len].  No column outside [0, leader_len) is ever read: a column index
 *       t + k past the end reads the last column leader_x[:, leader_len - 1] instead (a caller that wants the
 *       reference's window checks leader_len >= t + N + 1 up front).
 *   HVP_CENT_ADOPT (after the solve; reads u [S][n][N], modes [S][n][N], obj, status, nodes [S]): the rollout inputs
 *       u0 [S][n] = u[s][i][0] and, when gear0 is not NULL, gear0 [S][n] int32 = mode_gear[modes[s][i][0]] (mode
 *       index clamped to [0, n_modes)).  A scenario whose status is not 2 gets u0 = 0 and gear 6, as
 *       solve_mpc(raises=False) gives it.  For 0 <= t < T, row t of the episode logs: U_log [T][S][w] = u0, followed
 *       by the gears as doubles when gear0 is given (w = 2n: the reference's action [u_g ; gears]; else w = n);
 *       obj_log / status_log / nodes_log [T][S]; aborted_at [S] = the first t whose status is not 2 (-1: none; the
 *       row is reset at t == 0). */
#define HVP_CENT_PACK 0
#define HVP_CENT_ADOPT 1
typedef struct {
    int32_t n, N, S, phase;       /* phase: HVP_CENT_PACK | HVP_CENT_ADOPT */
    int32_t n_param;              /* PACK: length of a params row (hvp_mpc_info[2]), >= 2(N+1) */
    int32_t leader_per_scenario;  /* PACK: leader_x is [S][2][leader_len] (1) or [2][leader_len] shared (0) */
    int64_t leader_len;           /* PACK: columns of the leader trajectory (>= 1) */
    int64_t T;                    /* ADOPT: rows of the episode logs */
    int32_t n_modes;              /* ADOPT with gear0: entries of mode_gear (1..16) */
    int32_t reserved;
    int32_t mode_gear[16];        /* ADOPT with gear0: gear of each mode (hvp_mpc_mode_table) */
    const int64_t* t;             /* device pointer: timestep index */
    const double* leader_x;       /* PACK */
    double* params;               /* PACK: [S][n_param] */
    const double* u; const int32_t* modes; const double* obj; const int32_t* status; const int32_t* nodes; /* ADOPT in */
    double* u0; int32_t* gear0;   /* ADOPT out: [S][n] each; gear0 may be NULL */
    double* U_log; double* obj_log; int32_t* status_log; int32_t* nodes_log; int32_t* aborted_at;   /* ADOPT out */
} hvp_cent_step;
int hvp_cent_step_dev(hvp_ctx* ctx, const hvp_cent_step* g, void* stream);

/* ---- fused glue of an event-based iteration ------------------------------------------------------------------
 * What TrackingEventBasedCoordinator.get_control / on_timestep_end (fleet_event_based.py:42-107) do around the eval
 * and solve launches, for all S scenarios at once.  Agent i optimises its members m = [i-1, i, i+1] clipped at the
 * ends ([0, 1] for both agents when n = 2); agents with the same formulation form a group (one eval and one solve
 * launch each), whose rows are ordered [scenario][agent of the group]: agent i is row s * count + slot_of[i] of
 * group[group_of[i]], count = the number of agents with that group.  t is read from DEVICE memory.  Three phases:
 *   HVP_EVENT_PACK   (before the group launches; one thread per (scenario, agent)): x0[row][l] = x[s][m_l],
 *       xg[row][l] = SG[s][m_l], ug[row][l] = UG[s][m_l], and the parameter blocks [leader_x[:, t : t+N+1] if the
 *       group has a leader else 0 | SG[s][i-2] if i > 1 else 0 | SG[s][i+2] if i < n-2 else 0] (columns past the end
 *       of leader_x read its last column).  The rest of a params row is left alone.
 *   HVP_EVENT_SELECT (after the group launches; one warp per scenario; nothing for a scenario with active[s] == 0):
 *       cost0 = eval cost, cost1 = obj if status == 2 else +inf, dec = cost0 - cost1 (IEEE: inf - inf is NaN, never
 *       valid); the winner is the FIRST agent with the largest dec among those with dec > threshold.
 *       FEAS[t][s] &= any(isfinite(cost1)), ND[t][s] = max(ND[t][s], nodes of every agent), WIN[t][s][it] = winner or
 *       -1.  The winner's x / u (and, with GG, mode_gear[modes], mode index clamped to [0, n_modes)) overwrite
 *       SG / UG / GG of its members; no winner sets active[s] = 0 (the reference's `break`).
 *   HVP_EVENT_ADOPT  (after the last iteration, before the rollout; one thread per (scenario, agent)): u0 = UG[:, :, 0],
 *       gear0 = GG[:, :, 0] with gears, U_log[t] = u0 (then the gears as doubles: w = 2n), SG / UG / GG shifted one
 *       column left repeating the last one, active[s] = 1.
 * Log rows are written only for 0 <= t < T.  All pointers are device pointers. */
#define HVP_EVENT_PACK 0
#define HVP_EVENT_SELECT 1
#define HVP_EVENT_ADOPT 2
typedef struct {
    double* x0; double* xg; double* ug; double* params;  /* PACK out: [rows][nl][2], [rows][nl][2][N+1], [rows][nl][N], [rows][n_param] */
    const double* cost; /* SELECT in: eval output [rows] */
    const double* u; const double* x; const int32_t* modes; const double* obj; const int32_t* status; const int32_t* nodes; /* SELECT in: solve output */
    int32_t n_local;    /* members of each agent of the group (2 or 3) */
    int32_t n_param;    /* >= 6(N+1) */
    int32_t has_leader; /* the group's formulation has a relative leader (parameter block 0) */
    int32_t reserved;
} hvp_event_group;
typedef struct {
    int32_t n, N, S, phase;       /* phase: HVP_EVENT_PACK | HVP_EVENT_SELECT | HVP_EVENT_ADOPT */
    int32_t iters, it;            /* SELECT: iterations per timestep, this iteration (the WIN column) */
    int32_t ngroups;              /* 1..8 */
    int32_t leader_per_scenario;  /* PACK: leader_x is [S][2][leader_len] (1) or [2][leader_len] shared (0) */
    int64_t leader_len;           /* PACK: columns of the leader trajectory (>= 1) */
    int64_t T;                    /* SELECT / ADOPT: rows of the episode logs */
    double threshold;             /* SELECT: least cost decrease of a winner (exclusive) */
    int32_t n_modes;              /* SELECT with GG: entries of mode_gear (1..16) */
    int32_t reserved;
    int32_t mode_gear[16];
    int32_t group_of[64], slot_of[64];
    hvp_event_group group[8];
    const int64_t* t;             /* device pointer: timestep index */
    const double* x;              /* PACK: [S][n][2] */
    const double* leader_x;       /* PACK */
    double* SG; double* UG; int32_t* GG;   /* guesses [S][n][2][N+1], [S][n][N], [S][n][N] (GG NULL: pwa_gear) */
    uint8_t* active;              /* [S] */
    int32_t* WIN; uint8_t* FEAS; int32_t* ND;  /* SELECT logs [T][S][iters], [T][S], [T][S] */
    double* U_log;                /* ADOPT log [T][S][w] */
    double* u0; int32_t* gear0;   /* ADOPT out [S][n] each; gear0 with GG only */
} hvp_event_iter;
int hvp_event_iter_dev(hvp_ctx* ctx, const hvp_event_iter* g, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* HVP_H */
