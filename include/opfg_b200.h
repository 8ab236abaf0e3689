/*
 * opfg_b200.h -- C ABI of libopfg_b200.so: batched AC power flow + reward engine
 * for opfgym-style environments on NVIDIA B200 (sm_100a).
 *
 * Plain pointers and sizes only; no torch / C++ types cross this boundary.
 * Every `double*` / `uint8_t*` / `int32_t*` / `float*` argument of a launch
 * function is a DEVICE pointer unless its comment says "host".  All launches go
 * to the caller's `cudaStream_t` (passed as void*), never synchronise, and never
 * allocate.  Return value: 0 = ok, <0 = error (text via opfg_last_error()).
 * Non-convergence of an environment is DATA (converged[b] == 0), not an error.
 *
 * Which reference interface each entry point replaces
 * (paths relative to the opfgym reference checkout):
 *
 *   opfg_grid_create      pandapower `_pd2ppc`/`_ppc2ppci` output (`net._ppc`) consumed by
 *                         `pp.runpp`, reached from opfgym/opf_env.py:703; symbolic analysis
 *                         replaces SuperLU/KLU's per-call ordering.
 *   opfg_set_assembly     OpfEnv._apply_actions            opfgym/opf_env.py:421-491
 *                         + pandapower bus PD/QD summation (build_bus.py) [ext-mem]
 *   opfg_set_scoring      opfgym/constraints.py:70-128, opfgym/objective.py:6-87,
 *                         opfgym/reward.py:61-98, OpfEnv._get_obs opf_env.py:532-549
 *   opfg_philox_uniform   np_random.uniform in OpfEnv._sample_from_range  opf_env.py:278
 *   opfg_sample_uniform   OpfEnv._sample_uniform / _sample_from_range      opf_env.py:253-284
 *   opfg_sample_uniform_obs   ... with the reset observation written on the way   opf_env.py:218
 *   opfg_sample_profiles  OpfEnv._set_simbench_state (profile row, noise, clip)    opf_env.py:317-372
 *   opfg_assemble         OpfEnv._apply_actions + makeSbus (kernel 1)
 *   opfg_pf_solve         pp.runpp(net, enforce_q_lims=True)  opf_env.py:696-709
 *                         (kernels 2-4: mismatch SpMV, Jacobian, batched sparse LU)
 *   opfg_score            pfsoln/_extract_results + OpfEnv.calculate_reward opf_env.py:515-530
 *                         + OpfEnv._get_obs (kernel 5)
 *   opfg_step             OpfEnv.step                       opfgym/opf_env.py:374-419
 *   opfg_observe          OpfEnv._get_obs after reset       opfgym/opf_env.py:218, 532-549
 *   opfg_row_program_*    the `_sampling` overrides of the benchmark envs
 *                         (envs/voltage_control.py:121-133, load_shedding.py:131-149, ...)
 *   opfg_reset_plan_*,    OpfEnv.reset without a reset power flow (opf_env.py:180-220): sampler,
 *   opfg_reset_episode    hooks, initial action, _apply_actions, _get_obs in one launch
 *   opfg_set_dynamic_branches  pandapower's per-call branch / Ybus rebuild when trafo.tap_pos or
 *                         *.in_service are actions or contingencies
 *
 * opfg_pf_solve may issue two launches: the DC start of all environments as one FP64 GEMM
 * (B'^-1 is built at opfg_grid_create) and the persistent Newton-Raphson kernel; the `va` buffer
 * carries the start angles between them.
 */
#ifndef OPFG_B200_H
#define OPFG_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define OPFG_VERSION 1

/* PYPOWER column indices of the ppc matrices handed to opfg_grid_create */
enum { OPFG_BUS_I = 0, OPFG_BUS_TYPE = 1, OPFG_PD = 2, OPFG_QD = 3, OPFG_GS = 4, OPFG_BS = 5,
       OPFG_VM = 7, OPFG_VA = 8, OPFG_BASE_KV = 9 };
enum { OPFG_GEN_BUS = 0, OPFG_PG = 1, OPFG_QG = 2, OPFG_QMAX = 3, OPFG_QMIN = 4, OPFG_VG = 5,
       OPFG_GEN_STATUS = 7 };
enum { OPFG_F_BUS = 0, OPFG_T_BUS = 1, OPFG_BR_R = 2, OPFG_BR_X = 3, OPFG_BR_B = 4, OPFG_TAP = 8,
       OPFG_SHIFT = 9, OPFG_BR_STATUS = 10, OPFG_BR_G = 13 /* extension: shunt conductance */ };
enum { OPFG_PQ = 1, OPFG_PV = 2, OPFG_REF = 3 };

typedef struct OpfgGrid OpfgGrid; /* opaque; owns device copies of all tables */

/* ---- value references -------------------------------------------------------
 * Per-environment mutable cells live in one row-major state matrix S[B, n_state]
 * (sampled loads, set-points, prices, per-sample bounds ... and, at its tail,
 * the result cells written by opfg_score).  Static values shared by all
 * environments live in a constant table C[n_const].  A value reference is an
 * int32:  ref >= 0 -> S[b, ref];  ref < 0 -> C[-ref-1].                        */
typedef int32_t opfg_ref;
#define OPFG_NO_VM_REF ((opfg_ref)(-2147483647 - 1))

typedef struct {
    int32_t nb, ng, nbr;
    double base_mva;
    const double* bus;    int32_t bus_cols;     /* host, [nb , bus_cols]    row-major */
    const double* gen;    int32_t gen_cols;     /* host, [ng , gen_cols]              */
    const double* branch; int32_t branch_cols;  /* host, [nbr, branch_cols] (>=14 to carry BR_G) */
    double tol_pu;          /* ||F||_inf threshold, = tolerance_mva / base_mva          */
    int32_t max_iter;       /* pandapower max_iteration='auto' -> 10                      */
    int32_t init_dc;        /* 1: DC-power-flow angle start (pandapower init='dc')        */
    int32_t enforce_q_lims; /* 1: PV->PQ outer loop of pandapower's enforce_q_lims        */
    int32_t threads_per_env;/* 0 = choose from grid size (32/64/128)                      */
    int32_t ordering;       /* 0 = auto, 1 = min-degree, 2 = independent-set, 3 = least fill work;
                               auto roots each tree of a radial grid at its centre (fewest levels)   */
    int32_t pf_kernel;      /* 0 = auto, 1 = one CTA per environment (level-scheduled block LU in shared
                               memory), 2 = one LANE per environment (row-wise LU, Jacobian never stored,
                               state in global scratch), 3 = fused kernel for radial grids (8-32 lanes per
                               environment, Jacobian never stored, state in shared memory; auto picks it
                               when the grid is radial).  All three produce the same bits.               */
} OpfgGridDesc;

typedef struct {
    int32_t nb, n_nonref, nnz_y, n_blocks, n_fill_blocks, n_levels, threads_per_env;   /* n_blocks: 2x2 blocks of the FILLED Jacobian */
    int32_t smem_bytes_pf, smem_bytes_score;   /* per environment; _pf counts storage SLOTS (fill blocks reuse the slots of dead blocks) */
    int32_t n_state, n_const, n_act, n_obs, n_constraints;
    double flops_per_iter;     /* FP64 flops of one NR iteration (mismatch+Jacobian+LU+solves+update) */
    double flops_score;        /* FP64 flops of branch flows + scoring                                */
    double lu_flops;           /* block LU part of flops_per_iter                                     */
    double bytes_per_step;     /* algorithmic HBM bytes of one env step (see DESIGN.md)               */
    int32_t pf_kernel_used;    /* what opfg_pf_solve launches on this grid: 1 CTA per environment, 2 lane
                                  per environment, 3 fused kernel for radial grids                      */
    int32_t lane_max_row;      /* its largest row pattern (blocks) / warps per CTA / staged tables     */
    int32_t lane_warps_per_cta, lane_tables_staged;
    double lane_scratch_bytes; /* global scratch of the lane kernel (all resident warps)               */
    int32_t radial_lanes_per_env, radial_envs_per_cta, radial_smem_bytes_per_env;
    int32_t n_island_critical; /* dynamic branches whose outage can cut buses off (spanning-tree edges): only then
                                  does opfg_assemble walk the grid of an environment                     */
    int32_t cta_envs_per_cta;  /* CTA kernel: environments per CTA (1 = k_pf, one CTA per environment; > 1 = k_pf_multi) */
    int32_t cta_tables_staged; /* k_pf_multi: tables staged in shared memory, 0 = LU schedule + Ybus index tables,
                                  1 = + Ybus values, 2 = + start-value / DC / q-limit tables                  */
    int32_t score_threads_per_env; /* opfg_score: threads per environment (32 = k_score_warps, else k_score) */
} OpfgGridInfo;

/* action application + Sbus scatter (kernel 1) */
typedef struct {
    int32_t n_state;                 /* width of S                                   */
    int32_t n_const; const double* consts;           /* host, C table                */
    /* actions: S[slot] = round_kind(clamp(a*(hi-lo)+lo) / div) */
    int32_t n_act;
    const int32_t* act_slot;         /* host [n_act] S column written                 */
    const opfg_ref* act_lo;          /* host [n_act]                                  */
    const opfg_ref* act_hi;          /* host [n_act]                                  */
    const opfg_ref* act_div;         /* host [n_act] scaling divisor                  */
    const int32_t* act_kind;         /* host [n_act] 0 continuous, 1 bool round, 2 integer round */
    const opfg_ref* act_clamp_lo;    /* host [n_act] or NULL: clamp after mapping (non-autoscale mode) */
    const opfg_ref* act_clamp_hi;
    double act_diff_step;            /* > 0: incremental set-points (diff_action_step_size, opf_env.py:451-458):
                                        sp = (2a-1)*step*(hi-lo) + previous*div                             */
    /* injections: Sbus[bus] += coef * (P + jQ) / base_mva, in list order per bus */
    int32_t n_inj;
    const int32_t* inj_bus;          /* host [n_inj] ppc bus                           */
    const opfg_ref* inj_p;           /* host [n_inj]                                   */
    const opfg_ref* inj_q;           /* host [n_inj] (ref to a 0 constant if none)     */
    const opfg_ref* inj_coef;        /* host [n_inj] sign*scaling*in_service           */
    /* per-environment voltage set-points (gen.vm_pu / ext_grid.vm_pu as actions or sampled cells,
       reference anchor opfgym/envs/eco_dispatch.py:83): host [nb] by ppc bus, OPFG_NO_VM_REF where the
       bus keeps the static start value; NULL = all static.  opfg_assemble then writes the start |V| of
       every bus into the batch's `vm` buffer and opfg_pf_solve starts (and holds PV / slack buses) there. */
    const opfg_ref* bus_vm_ref;
} OpfgAssemblyDesc;

enum { OPFG_REWARD_SUMMATION = 0, OPFG_REWARD_REPLACEMENT = 1, OPFG_REWARD_PARAMETERIZED = 2,
       OPFG_REWARD_ONLY_OBJECTIVE = 3 };

/* result cells, constraints, costs, reward, observation gather (kernel 5) */
typedef struct {
    int32_t n_inputs;                /* S[:, n_inputs:] are result cells (written by opfg_score) */
    /* where results go in S (-1 = not materialised) */
    int32_t n_pp_bus;
    const int32_t* pp_bus_lookup;    /* host [n_pp_bus] pandapower bus -> ppc bus (-1 dropped) */
    int32_t res_bus_vm_slot, res_bus_va_slot;        /* first S column of res_bus.vm_pu / va_degree */
    const int32_t* branch_loading_slot;              /* host [nbr] S column of loading_percent (-1 none) */
    const int32_t* branch_flow_slot;                 /* host [nbr] first of 4 S columns p_from,q_from,p_to,q_to (-1) */
    const double* rate_f; const double* rate_t;      /* host [nbr] loading = 100*max(|Sf|*rate_f/vm_f, |St|*rate_t/vm_t) */
    const int32_t* gen_p_slot; const int32_t* gen_q_slot; /* host [ng] S columns of generator P/Q results (-1) */
    /* constraints */
    int32_t n_constraints;
    const int32_t* con_ptr;          /* host [n_constraints+1] element ranges          */
    const opfg_ref* con_value;       /* host [n_el]                                    */
    const double*  con_value_scale;  /* host [n_el]                                    */
    const opfg_ref* con_min;         /* host [n_el] (ref to NaN constant = unbounded)  */
    const opfg_ref* con_max;         /* host [n_el]                                    */
    const double*  con_bound_mul;    /* host [n_el] boundary multiplier (scaling)      */
    const double*  con_autoscale;    /* host [n_constraints]                           */
    const int32_t* con_worst_case;   /* host [n_constraints]                           */
    const double*  con_penalty_factor; const double* con_penalty_power; const double* con_count_penalty;
    /* polynomial costs: cost = c0 + c1*v + c2*v^2 for P and for Q of each row */
    int32_t n_poly;
    const opfg_ref* poly_p; const double* poly_p_mul;   /* host [n_poly] P value = mul * ref */
    const opfg_ref* poly_q; const double* poly_q_mul;
    const opfg_ref* poly_coef;       /* host [n_poly*6] cp0 cp1 cp2 cq0 cq1 cq2        */
    /* piece-wise linear costs */
    int32_t n_pwl, n_pwl_seg;        /* every row uses the first n_pwl_seg segments    */
    const opfg_ref* pwl_v; const double* pwl_v_mul;     /* host [n_pwl]                */
    const opfg_ref* pwl_seg;         /* host [n_pwl*n_pwl_seg*3] lo, hi, price         */
    /* reward */
    int32_t reward_kind;
    double penalty_weight;           /* NaN = None (plain sum)                         */
    double clip_lo, clip_hi;         /* NaN = no clipping                              */
    double objective_factor, objective_bias, penalty_factor, penalty_bias;
    double valid_reward, invalid_penalty, invalid_objective_share;
    /* observation gather */
    int32_t n_obs;
    const opfg_ref* obs_ref;         /* host [n_obs], or [obs_ptr[n_obs]] with obs_ptr  */
    const int32_t* obs_ptr;          /* host [n_obs+1] or NULL: observation j is the SUM of
                                        obs_ref[obs_ptr[j] .. obs_ptr[j+1]) (bus_wise_obs,
                                        opf_env.py:535-536, 806-810)                    */
    /* three-winding transformers (net.trafo3w): three branch rows each, hv->star, star->mv, star->lv, whose
       branch_loading_slot entries point at three consecutive result cells and whose rate_f / rate_t are 0 at the
       star end, so that each cell holds the loading at the outer end of its row.  Kernel 5 then writes
       res_trafo3w.loading_percent = the largest of the three, NaN if any of them is NaN.
       n_trafo3w = 0: none (the pointers may be NULL). */
    int32_t n_trafo3w;
    const int32_t* trafo3w_row_slot;     /* host [n_trafo3w] first of the 3 S columns of the rows' loadings (hv, mv, lv) */
    const int32_t* trafo3w_loading_slot; /* host [n_trafo3w] S column of res_trafo3w.loading_percent                     */
} OpfgScoringDesc;

/* per-environment branch parameters (tap_pos / in_service actions, N-1 contingencies): the listed
 * branches get their admittances -- and Ybus its values -- recomputed per environment by
 * opfg_assemble (kernel 1), in the fixed sparsity pattern of the nominal topology.
 * Replaces pandapower's per-call `_calc_branch_values_from_trafo_df` / `_calc_line_parameter` +
 * makeYbus for those branches (reached from opfgym/opf_env.py:476-483, 703).
 * Islands: if a cleared in-service cell cuts buses off every reference bus, opfg_assemble finds them per
 * environment (pandapower pd2ppc `_check_connectivity`: such buses are dropped from the power flow) and
 * opfg_pf_solve solves the rest; `vm` / `va` of a dropped bus come back NaN, `converged` stays 1. */
typedef struct {
    int32_t n_dyn;
    const int32_t* branch;          /* host [n_dyn] ppc branch row                                        */
    const opfg_ref* tap_pos;        /* host [n_dyn] tap position cell (ref to a NaN constant: tap fixed)   */
    const double* tap_neutral;      /* host [n_dyn]                                                        */
    const double* tap_step_percent; /* host [n_dyn]                                                        */
    const double* ratio_neutral;    /* host [n_dyn] off-nominal ratio at the neutral tap (HV-side changer) */
    const opfg_ref* in_service;     /* host [n_dyn] 0/1 cell (ref to constant 1: always in service)        */
    /* optional, NULL = absent.  Switches at the branch ends (`switch.closed` of line-bus / trafo-bus switches,
     * opfgym/examples/network_reconfiguration.py:34, security_constrained.py:31): a transformer with an open
     * switch is out of service; a line that is open at ONE end stays energised from the other end (pandapower
     * inserts an auxiliary bus there; here that bus is eliminated analytically), open at both ends it is out. */
    const opfg_ref* closed_from;    /* host [n_dyn] 0/1 cell of the switch at the from / hv end (ref to constant 1: none) */
    const opfg_ref* closed_to;      /* host [n_dyn] ... at the to / lv end                                  */
    const int32_t* flags;           /* host [n_dyn] OPFG_DYN_* bits                                        */
} OpfgDynBranchDesc;
enum { OPFG_DYN_TAP_LV = 1,         /* tap changer on the LV side: ratio / t, series impedance * t^2, magnetising branch / t^2 */
       OPFG_DYN_TRAFO = 2,          /* transformer: any open switch takes it out of service                 */
       OPFG_DYN_NORMALLY_OPEN = 4 };/* hint: out of service / open in the nominal topology (a tie).  The spanning tree that decides
                                       which outages can island anything is grown through the other branches first */

/* device buffers of one batch (any pointer may be NULL if the stage that needs it is not run) */
typedef struct {
    int64_t n_env;
    const double* actions;   /* [B, n_act]   in  (opfg_assemble; NULL = keep set-points, Sbus only)   */
    double* state;           /* [B, n_state] in/out                                           */
    double* sbus;            /* [B, nb, 2]   complex bus injections, ppc bus order, p.u.
                                (opfg_assemble: NULL = write the set-points only)            */
    double* vm;              /* [B, nb]      out, p.u.                                        */
    double* va;              /* [B, nb]      out, radians                                     */
    uint8_t* converged;      /* [B]          out                                              */
    int32_t* iterations;     /* [B]          out                                              */
    double* reward;          /* [B]          out (NaN if not converged)                       */
    double* objective;       /* [B]          out  sum of -costs                               */
    double* penalty;         /* [B]          out  sum of penalties                            */
    double* cost;            /* [B]          out  safe-RL cost                                */
    uint8_t* valids;         /* [B, n_constraints] out                                        */
    double* violations;      /* [B, n_constraints] out                                        */
    double* penalties;       /* [B, n_constraints] out                                        */
    float*  obs_f32;         /* [B, n_obs] out (either or both)                               */
    double* obs_f64;         /* [B, n_obs] out                                                */
    double* stats;           /* [OPFG_N_STATS] accumulated with atomics; caller zeroes        */
    double* yval;            /* [B, nnz_y, 2] per-env Ybus values, only with dynamic branches  */
    double* bry;             /* [B, n_dyn, 8] per-env admittances of the dynamic branches      */
    const double* objective_offset; /* [B] or NULL: subtracted from the objective (diff_objective,
                                       opf_env.py:497-498: -costs - initial_obj)                    */
    int32_t absolute_actions;       /* != 0: kernel 1 ignores act_diff_step (reset applies the initial
                                       action as an absolute set-point, opf_env.py:207)             */
    int32_t stats_slots;            /* > 1: `stats` is [stats_slots][OPFG_N_STATS] and environment b adds to
                                       row b % stats_slots (the caller sums the rows); thousands of
                                       atomics on ONE row serialise in L2 (0.11 ms of kernel 5 at 32 768 envs) */
} OpfgBatch;

enum { OPFG_STAT_N = 0, OPFG_STAT_CONVERGED = 1, OPFG_STAT_VALID = 2, OPFG_STAT_SUM_REWARD = 3,
       OPFG_STAT_SUM_REWARD_SQ = 4, OPFG_STAT_SUM_OBJECTIVE = 5, OPFG_STAT_SUM_PENALTY = 6,
       OPFG_STAT_SUM_ITERS = 7, OPFG_STAT_VIOLATED0 = 8 /* +c: envs violating constraint c */,
       OPFG_N_STATS = 24 };

int         opfg_version(void);
const char* opfg_last_error(void);

int  opfg_grid_create(const OpfgGridDesc* desc, OpfgGrid** out);
void opfg_grid_destroy(OpfgGrid* grid);
int  opfg_set_assembly(OpfgGrid* grid, const OpfgAssemblyDesc* desc);
int  opfg_set_scoring(OpfgGrid* grid, const OpfgScoringDesc* desc);
int  opfg_set_dynamic_branches(OpfgGrid* grid, const OpfgDynBranchDesc* desc);   /* after opfg_set_assembly */
int  opfg_grid_info(const OpfgGrid* grid, OpfgGridInfo* out);
/* host copies of the symbolic analysis, for inspection/tests: perm[n_nonref] = ppc bus of pivot k,
 * level_ptr[n_levels+1]; either pointer may be NULL */
int  opfg_grid_symbolic(const OpfgGrid* grid, int32_t* perm, int32_t* level_ptr);

/* out[b, j] = U[0,1) double from Philox4x32-10, key = seed, counter = (j/2, first_env + b, stream);
 * independent of how environments are sharded over GPUs */
int opfg_philox_uniform(uint64_t seed, uint64_t first_env, uint64_t stream_id,
                        int64_t n_env, int32_t n_cols, double* out, void* cuda_stream);

/* OpfEnv._sample_from_range (opfgym/opf_env.py:266-284), fused with the generator:
 * state[b, slots[j]] = (lo[j] + (hi[j] - lo[j]) * u(b, j)) / div[j], u as in opfg_philox_uniform.
 * slots / lo / hi / div are DEVICE arrays of length n_cols. */
int opfg_sample_uniform(uint64_t seed, uint64_t first_env, uint64_t stream_id, int64_t n_env,
                        int32_t n_cols, const int32_t* slots, const double* lo, const double* hi,
                        const double* div, double* state, int32_t n_state, void* cuda_stream);
/* The same, and the sampled values go straight into the observation as well (OpfEnv._get_obs after reset,
 * opf_env.py:218, 532-549, when the observed cells are exactly cells this sampler writes): obs_pos[j] = position of
 * column j in the observation row or -1; exactly one of obs_f32 / obs_f64 ([n_env, n_obs]) is given.  Saves
 * re-reading the state row for the reset observation (opfg_observe). */
int opfg_sample_uniform_obs(uint64_t seed, uint64_t first_env, uint64_t stream_id, int64_t n_env,
                            int32_t n_cols, const int32_t* slots, const double* lo, const double* hi,
                            const double* div, double* state, int32_t n_state, const int32_t* obs_pos,
                            float* obs_f32, double* obs_f64, int32_t n_obs, void* cuda_stream);

/* OpfEnv._set_simbench_state (opf_env.py:317-372; the reference's DEFAULT sampler, train_data='simbench'):
 * S[b, slots[j]] = clip(noise(table[step[b], j] (optionally interpolated towards step + 1 with interp_r[b])),
 * pmin[j], pmax[j]).  noise_kind 0 none, 1 uniform (value * U(1 - f, 1 + f)), 2 normal (value + |value| f N(0,1)).
 * table: device [n_steps, n_cols] row-major (one profile table = one element table's column); step: device
 * int64 [n_env]; random numbers are Philox rows keyed like opfg_philox_uniform (uniform: n_cols wide,
 * normal: 2 n_cols wide). */
int  opfg_sample_profiles(uint64_t seed, uint64_t first_env, uint64_t stream_id, int64_t n_env, int32_t n_cols,
                          const int32_t* slots, const double* table, int32_t n_steps, const int64_t* step,
                          const double* interp_r /* device [n_env] or NULL */, const double* pmin,
                          const double* pmax, double noise_factor, int32_t noise_kind, double* state,
                          int32_t n_state, void* cuda_stream);

int opfg_assemble(const OpfgGrid* grid, const OpfgBatch* batch, void* cuda_stream);
int opfg_pf_solve(const OpfgGrid* grid, const OpfgBatch* batch, void* cuda_stream);
int opfg_score(const OpfgGrid* grid, const OpfgBatch* batch, void* cuda_stream);
/* observation gather only (OpfEnv._get_obs after reset, opf_env.py:218): obs[b, j] = value(obs_ref[j]) */
/* ---- mixed batch (BASELINE.json configs[3]: "MaxRenewable + QMarket mixed batch, fused constraint /
 * objective / reward kernel"): environments of SEVERAL grids scored by ONE launch of kernel 5 (and assembled by
 * one launch of kernel 1).  Every CTA picks its member's descriptor and batch from a device table by its
 * block index.  The power flows in between stay per member (opfg_pf_solve; different kernels per grid size).
 * Reference hooks the single launch carries: envs/max_renewable.py:93-105, envs/voltage_control.py:105-133. */
typedef struct OpfgMixed OpfgMixed;
int  opfg_mixed_create(int32_t n_members, const OpfgGrid* const* grids, const OpfgBatch* batches /* host [n] */,
                       OpfgMixed** out);
void opfg_mixed_destroy(OpfgMixed* mixed);
int  opfg_assemble_mixed(OpfgMixed* mixed, const OpfgBatch* batches /* host [n], re-read every call */, void* cuda_stream);
int  opfg_score_mixed(OpfgMixed* mixed, const OpfgBatch* batches /* host [n] */, void* cuda_stream);

int opfg_observe(const OpfgGrid* grid, const OpfgBatch* batch, void* cuda_stream);
/* assemble -> pf_solve -> score, back to back on the stream */
int opfg_step(const OpfgGrid* grid, const OpfgBatch* batch, void* cuda_stream);

/* ---- per-row column programs -------------------------------------------------------------
 * The env `_sampling` hooks of the reference (opfgym/envs/voltage_control.py:121-133,
 * load_shedding.py:131-149, max_renewable.py:101-105 ...) derive per-sample bounds and prices
 * row by row from sampled columns.  A row program runs, for every environment and every row of
 * one table, a short list of ops on 16 f64 registers -- one launch per hook. */
enum { OPFG_OP_LOAD_STATE = 0 /* r[dst] = S[b, a + row] */, OPFG_OP_LOAD_STATIC = 1 /* r[dst] = statics[a + row] */,
       OPFG_OP_CONST = 2 /* r[dst] = imm */, OPFG_OP_ADD = 3, OPFG_OP_SUB = 4, OPFG_OP_MUL = 5, OPFG_OP_DIV = 6,
       OPFG_OP_SQRT = 7 /* r[dst] = sqrt(r[a]) */, OPFG_OP_NEG = 8, OPFG_OP_MIN = 9, OPFG_OP_MAX = 10,
       OPFG_OP_ABS = 11, OPFG_OP_STORE_STATE = 12 /* S[b, a + row] = r[b] */ };
typedef struct { int32_t op, dst, a, b; double imm; } OpfgRowOp;
typedef struct OpfgRowProgram OpfgRowProgram;
int  opfg_row_program_create(int32_t n_rows, int32_t n_ops, const OpfgRowOp* ops /* host */,
                             int32_t n_static, const double* statics /* host */, OpfgRowProgram** out);
void opfg_row_program_destroy(OpfgRowProgram* program);
/* Run the program on a subset of the table's rows only (host array of row numbers): rows whose stores
 * no kernel table ever reads need not be computed (row-level pruning by the table compiler). */
int  opfg_row_program_select_rows(OpfgRowProgram* program, int32_t n_selected, const int32_t* rows /* host */);
/* Fails, launching nothing, if a state cell the program touches on one of its rows is >= n_state. */
int  opfg_row_program_run(const OpfgRowProgram* program, int64_t n_env, double* state, int32_t n_state,
                          void* cuda_stream);

/* ---- fused episode reset ---------------------------------------------------------------------
 * OpfEnv.reset (opfgym/opf_env.py:180-220) for `full_uniform` data without a reset power flow:
 * `_sampling` (sampler stages and hook row programs, in the order the env issues them), the initial
 * action (centre or random, :201-207), `_apply_actions` and `_get_obs` -- ONE launch, one CTA per
 * environment; the state row is written once and the observation comes out of the same pass.
 * Results are bit-identical to the sequence opfg_sample_uniform / opfg_row_program_run /
 * opfg_philox_uniform / opfg_assemble / opfg_observe with stream ids `stream_base + stream_offset`. */
typedef struct {
    int32_t kind;                    /* 0: uniform sampler stage, 1: row program stage            */
    int32_t n_cols;                  /* kind 0                                                    */
    const int32_t* slots;            /* kind 0, DEVICE [n_cols]                                   */
    const double* lo;                /* kind 0, DEVICE [n_cols]                                   */
    const double* hi;
    const double* div;
    uint32_t stream_offset;          /* kind 0: Philox stream = stream_base + stream_offset       */
    const OpfgRowProgram* program;   /* kind 1                                                    */
} OpfgResetStage;
typedef struct OpfgResetPlan OpfgResetPlan;
int  opfg_reset_plan_create(const OpfgResetStage* stages /* host */, int32_t n_stages, OpfgResetPlan** out);
void opfg_reset_plan_destroy(OpfgResetPlan* plan);
/* batch needs state, actions (receives the initial action) and an obs buffer.
 * random_action: 0 = centre action 0.5, 1 = U[0,1) from Philox stream stream_base + action_stream_offset */
int  opfg_reset_episode(const OpfgGrid* grid, const OpfgBatch* batch, const OpfgResetPlan* plan,
                        uint64_t seed, uint64_t first_env, uint64_t stream_base, int32_t random_action,
                        uint32_t action_stream_offset, void* cuda_stream);

/* FP64 FMA throughput probe for the roofline denominator (MEASURED_PEAKS.json has no FP64 figure):
 * every thread runs 8 independent DFMA chains of `iters` steps; flops = 2*8*iters*n_blocks*256.
 * out (device, >= 1 double) keeps the result alive. */
int opfg_fp64_probe(int32_t n_blocks, int32_t iters, double* out, void* cuda_stream);

/* number of kernel launches issued by this library since load (for bench accounting) */
int64_t opfg_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* OPFG_B200_H */
