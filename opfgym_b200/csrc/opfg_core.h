// Per-environment algorithms of the engine, written once and compiled twice:
//   * by nvcc for sm_100a (the product: one CTA per environment, working set in
//     shared memory, warp-shuffle reductions) and
//   * by g++ with -DOPFG_HOSTSIM into tests/hostsim/libopfg_hostsim.so, where one
//     host "thread" (tid 0 of 1) walks the same tables.  The host build exists so
//     that the symbolic schedule and the table marshalling can be unit-tested on
//     the GPU-less builder box; it is NOT reachable from the product package.
#pragma once
#include <cmath>
#include <cstdint>

#include "../../include/opfg_b200.h"

#if defined(__CUDACC__) && !defined(OPFG_HOSTSIM)
#define OPFG_DEVICE_BUILD 1
#define OPFG_HD __device__ __forceinline__
#define OPFG_HHD __host__ __device__ __forceinline__
#else
#define OPFG_HD inline
#define OPFG_HHD inline
#endif

namespace opfg {

struct U2 { uint32_t x, y; };

struct GridDev {
    // sizes
    int nb, n, n_levels, n_blocks, n_fill, nnz_y, nbr, ng, n_ref;
    int threads;
    double base_mva, tol;
    int max_iter, init_dc;
    int dc_pre;                        // 1: the DC start comes from the dense pre-pass (k_dc_start) through va
    const double* dc_binv_t;           // [n_pad_k][n_pad_i] transpose of B'^-1, zero padded (pre-pass)
    const double* dc_theta0;           // [n] B'^-1 * (constant part of the DC right-hand side)
    int dc_ld;                         // leading dimension (n_pad_i) of dc_binv_t
    // numbering
    const int* bus_of_int;
    const int* int_of_bus;
    const unsigned char* type_int;     // bus type by internal index
    const double* vm0_int;             // start |V| (init_vm_pu, or the set-point at generator buses)
    const double* va0_int;             // start angle (rad); ref buses keep it
    // schedule
    const int* level_ptr;
    const int* fill_ids;
    // packed 16-bit block / pivot ids (n_blocks, nb < 65536 is checked at grid creation)
    const int* dp_ptr;                 // [n+1] pair ranges of the diagonal items
    const U2* dp_pack;                 // {l | w<<16, m}
    const int* dp_own;                 // [n] first pair of the pivot's own item (sources one level below)
    const int* eg_ptr;                 // [n_levels+1] eager gather items per diagonal phase
    const U2* eg_item;                 // {k | n_pairs<<16, first pair}
    const int* off_ptr;                // [n_levels+1] off-diagonal item ranges
    const U2* off_hdr;                 // [n_items+1] {tgt | (piv+1)<<16, first pair}; last entry = sentinel
    const uint32_t* op_pack;           // l | w<<16
    const int* up_ptr;                 // [n+1]
    const uint32_t* up_pack;           // w | j<<16
    // Ybus
    const int *y_ptr, *y_diag;
    const U2* y_meta;                  // {col | (jacobian block + 1)<<16, row}
    int nnz_y_nonref;                  // entries of the non-slack rows come first
    const double* y_val;               // [nnz_y*2] re,im  (written by the Ybus assembly kernel)
    const int *yc_ptr, *yc_branch, *yc_role;
    const double* br_param;            // [nbr*6] r x b g tap shift_rad  (ppc branch table)
    double* br_y;                      // [nbr*8] Yff Yft Ytf Ytt (re,im)
    const double* bus_ysh;             // [nb*2] (GS + jBS)/base by ppc bus
    const int* br_f;                   // [nbr] ppc from bus
    const int* br_t;
    // enforce_q_lims: PV buses whose generators have active reactive limits (a generator with a zero
    // limit is skipped like pandapower does); limits are per bus, in p.u. of base_mva
    int n_qlim;
    const int* qlim_bus;               // [n_qlim] internal bus index
    const double *qlim_min, *qlim_max; // [n_qlim]
    // per-environment branch parameters (tap / in-service cells): kernel 1 rebuilds their
    // admittances and the Ybus values per environment
    int n_dyn;
    const int* dyn_branch;             // [n_dyn] ppc branch row
    const int* dyn_of_branch;          // [nbr] index into the dynamic list or -1
    const int *dyn_tap_ref, *dyn_svc_ref;
    const int *dyn_cf_ref, *dyn_ct_ref;          // switches at the from / to end (reference to constant 1: none)
    const int* dyn_flags;                        // OPFG_DYN_* bits
    const double *dyn_neutral, *dyn_step, *dyn_ratio0;
    const double* dyn_lv_scale;                  // LV-side tap changers: 1 / t0^2 (the branch row was built at the static tap t0)
    // islands: an in-service cell that is 0 can cut buses off every slack bus.  pandapower drops them
    // (pd2ppc.py _check_connectivity [ext-mem]: bus type NONE, results NaN) and solves the rest.  Kernel 1
    // finds them per environment -- only when a branch of the static grid's spanning tree is out, `dyn_crit` --
    // and marks them with a start |V| of exactly 0; the power-flow kernels keep such a bus at V = 0 behind
    // identity Jacobian rows (same linear system as the reduced grid) and report NaN for it.
    int isl;
    const unsigned char* dyn_crit;     // [n_dyn] 1: the branch is a spanning-tree edge
    const int *isl_ptr, *isl_adj, *isl_br;   // CSR by ppc bus over the branches that can be in service: neighbour bus, branch row
    // ---- assembly (kernel 1) ----
    int n_state, n_const, n_act, n_inj;
    double act_diff_step;
    const double* consts;
    const double* consts_end;          // one past a back-to-front copy of the constants: consts_end[r] = consts[-r-1], r < 0
    const int* act_slot;
    const int *act_lo, *act_hi, *act_div, *act_kind, *act_clamp_lo, *act_clamp_hi;
    const int* inj_ptr;                // [nb+1] CSR by ppc bus
    const int* inj_order;              // [nb] buses sorted by descending entry count
    const int *inj_p, *inj_q, *inj_coef;
    // per-environment voltage set-points (gen.vm_pu / ext_grid.vm_pu as state cells): kernel 1 writes the
    // start |V| of every bus into the `vm` buffer, the power-flow kernels start from there
    int vm_from_state;
    const int* bus_vm_ref;             // [nb] ppc bus -> value reference, or OPFG_NO_REF
    const double* vm0_bus;             // [nb] default start |V| by ppc bus
    // ---- scoring (kernel 5) ----
    int n_pp_bus, res_vm_slot, res_va_slot;
    const int* pp_lookup;
    const int *br_loading_slot, *br_flow_slot;
    const double *rate_f, *rate_t;
    int n_t3;                          // three-winding transformers (OpfgScoringDesc.trafo3w_*)
    const int *t3_row_slot, *t3_loading_slot;
    const int *gen_bus, *gen_p_slot, *gen_q_slot;
    const double* gen_q_share;
    int n_con;
    const int* con_ptr;
    const int *con_value, *con_min, *con_max;
    const double *con_value_scale, *con_bound_mul, *con_autoscale, *con_pfactor, *con_ppower, *con_pcount;
    const int* con_worst;
    int n_poly, n_pwl, n_pwl_seg;
    const int *poly_p, *poly_q, *poly_coef, *pwl_v, *pwl_seg;
    const double *poly_p_mul, *poly_q_mul, *pwl_v_mul;
    int reward_kind;
    double penalty_weight, clip_lo, clip_hi, obj_factor, obj_bias, pen_factor, pen_bias;
    double valid_reward, invalid_penalty, invalid_obj_share;
    int n_obs;
    const int* obs_ref;
    const int* obs_ptr;      // nullptr: one ref per observation
    int n_obs_runs;          // > 0: the observation is a few runs of consecutive state cells
    const int* obs_runs;     // [n_obs_runs][3] first state cell, first observation entry, length
    // ---- lane-per-environment power flow (row-wise schedule, symbolic.hpp LaneSchedule) ----
    int ln_max_row, ln_n_up;
    const int* ln_row;                 // [n+1][4] first Ybus entry, fill position, elimination item, upper block of row k
    const uint32_t* ln_y;              // [nnz_y_nonref] column | (row-buffer position + 1) << 16
    const unsigned char* ln_diag_pos;  // [n]
    const unsigned char* ln_fill;      // row-buffer positions that start at zero
    const uint32_t* ln_el;             // elimination items: position of L(k, m) | m << 16
    const int* ln_el_uptr;             // their update ranges
    const uint32_t* ln_upd;            // updates: W slot | target position << 16
    const uint32_t* ln_up;             // upper blocks: column j | position << 16
    const char* tab3_base;             // arena of the tables above (+ the Ybus values / start values they need)
    int tab3_bytes;
    const double* ln_yval;             // copies inside the lane arena
    const double *ln_vm0, *ln_va0;
    const int* ln_bus_of_int;
    const unsigned char* ln_type;
    const int* ln_qbus;                // q-limit tables (copies of qlim_*)
    const double *ln_qmin, *ln_qmax;
    // ---- fused kernel for radial grids (every pivot has at most one later neighbour) ----
    int tr_ok;
    const int *tr_bus_of_int, *tr_level_ptr, *tr_y_ptr, *tr_parent;
    const unsigned char* tr_type;
    const uint32_t* tr_y_ent;          // per Ybus entry: column | kind << 16 (0 other, 1 child, 2 parent)
    const double *tr_y_val, *tr_vm0, *tr_va0;
    const char* tab4_base;
    int tab4_bytes;
    const char* tab_base;              // contiguous arena holding the power-flow tables
    int tab_bytes;
    int tab_hot_bytes;                 // prefix holding the LU schedule
    int tab_warm_bytes;                // ... plus the Ybus tables (start values / DC factor / q-limits follow)
    int tab_staged_bytes;              // how much of the arena the multi-environment kernel stages
    const char* tab2_base;             // contiguous arena holding the scoring tables
    int tab2_bytes;
    int n_inputs;                      // S[:, n_inputs:] are the result cells written by kernel 5
    unsigned long long* phase_cycles;  // developer instrumentation (OPFG_PHASE_TIMING builds), else unused
};

// ------------------------------------------------------------------ block context
#ifdef OPFG_DEVICE_BUILD
template <int T>
struct Ctx {
    int tid;
    double* red;   // shared scratch, >= T/32 doubles
    int bar_id;    // 0: the environment owns the CTA; >0: named barrier of this environment's T threads
    __device__ __forceinline__ int nthreads() const { return T; }
    __device__ __forceinline__ void sync() const {
        if (T == 32) __syncwarp();
        else if (bar_id) asm volatile("bar.sync %0, %1;" ::"r"(bar_id), "n"(T) : "memory");
        else __syncthreads();
    }
    __device__ __forceinline__ double warp_max(double v) const {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
        return v;
    }
    __device__ __forceinline__ double warp_sum(double v) const {
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        return v;
    }
    // NaN-propagating max over the block (fmax would drop NaNs: carry a flag)
    __device__ __forceinline__ double block_max(double v) const {
        double bad = (v != v) ? 1.0 : 0.0;
        v = warp_max(bad > 0 ? 0.0 : v);
        bad = warp_max(bad);
        if (T > 32) {
            sync();
            if ((tid & 31) == 0) { red[tid >> 5] = v; red[(T >> 5) + (tid >> 5)] = bad; }
            sync();
            v = red[0]; bad = red[T >> 5];
#pragma unroll
            for (int w = 1; w < (T >> 5); ++w) { v = fmax(v, red[w]); bad = fmax(bad, red[(T >> 5) + w]); }
            sync();
        }
        return bad > 0 ? NAN : v;
    }
    __device__ __forceinline__ double block_sum(double v) const {
        v = warp_sum(v);
        if (T > 32) {
            sync();
            if ((tid & 31) == 0) red[tid >> 5] = v;
            sync();
            v = 0;
#pragma unroll
            for (int w = 0; w < (T >> 5); ++w) v += red[w];
            sync();
        }
        return v;
    }
};
#else
template <int T>
struct Ctx {
    int tid = 0;
    double* red = nullptr;
    int bar_id = 0;
    int nthreads() const { return 1; }
    void sync() const {}
    double block_max(double v) const { return v; }
    double block_sum(double v) const { return v; }
};
#endif

#if defined(OPFG_PHASE_TIMING) && defined(OPFG_DEVICE_BUILD)
#define OPFG_TICK(slot) do { if (cx.tid == 0 && g.phase_cycles) { const long long now_ = clock64(); \
    atomicAdd(g.phase_cycles + (slot), (unsigned long long)(now_ - tick_)); tick_ = now_; } } while (0)
#define OPFG_TICK_INIT long long tick_ = clock64()
#else
#define OPFG_TICK(slot) do {} while (0)
#define OPFG_TICK_INIT do {} while (0)
#endif

// value of a reference: state cell (r >= 0) or constant (r < 0); one load behind a selected
// address, so lanes holding different kinds of reference do not diverge
OPFG_HD double ref_val(const GridDev& g, const double* S, int r) {
    // constants are ALSO stored back to front, ending at consts_end: C[-r-1] == consts_end[r].  Only the base
    // depends on the kind of reference then, the index is r itself (two instructions fewer per reference)
    const double* base = r >= 0 ? S : g.consts_end;
    return base[r];
}

constexpr int OPFG_NO_REF = -2147483647 - 1;

// ------------------------------------------------- kernel 1a: branch -> Ybus values
// Admittances of one branch from its ppc row (pypower makeYbus.py [ext-mem]).
OPFG_HD void branch_admittance(const double* p, double* y) {
    const double r = p[0], x = p[1], b = p[2], gsh = p[3];
    double tap = p[4];
    const double sh = p[5];
    if (tap == 0.0) tap = 1.0;
    const double z2 = r * r + x * x;
    const double ysr = r / z2, ysi = -x / z2;
    const double ttr = ysr + 0.5 * gsh, tti = ysi + 0.5 * b;
    double c = 1.0, s = 0.0;                                  // lines and most transformers: no phase shift
    if (sh != 0.0) { c = cos(sh); s = sin(sh); }
    const double t2 = tap * tap;
    y[0] = ttr / t2;  y[1] = tti / t2;                        // Yff = Ytt / |tap|^2
    // Yft = -Ys / conj(tap) = -Ys * tap / |tap|^2 ; tap = tap*(c + js)
    y[2] = -(ysr * c - ysi * s) / tap;  y[3] = -(ysr * s + ysi * c) / tap;
    // Ytf = -Ys / tap = -Ys * conj(tap) / |tap|^2
    y[4] = -(ysr * c + ysi * s) / tap;  y[5] = -(-ysr * s + ysi * c) / tap;
    y[6] = ttr;  y[7] = tti;
}

// one Ybus CSR entry = ordered sum of its branch / shunt contributions
OPFG_HD void ybus_entry(const GridDev& g, const double* br_y, int e, double* out,
                        const double* bry_env = nullptr) {
    double re = 0, im = 0;
    for (int c = g.yc_ptr[e]; c < g.yc_ptr[e + 1]; ++c) {
        const int role = g.yc_role[c], idx = g.yc_branch[c];
        if (role == 4) { re += g.bus_ysh[2 * idx]; im += g.bus_ysh[2 * idx + 1]; continue; }
        const double* y = br_y + 8 * idx;
        if (bry_env) { const int d = g.dyn_of_branch[idx]; if (d >= 0) y = bry_env + 8 * d; }
        re += y[2 * role]; im += y[2 * role + 1];
    }
    out[0] = re; out[1] = im;
}

// observation j: one cell, or the sum of a group of cells (bus_wise_obs, opf_env.py:806-810)
OPFG_HD double obs_value(const GridDev& g, const double* S, int j) {
    if (!g.obs_ptr) return ref_val(g, S, g.obs_ref[j]);
    double v = 0.0;
    for (int k = g.obs_ptr[j]; k < g.obs_ptr[j + 1]; ++k) v += ref_val(g, S, g.obs_ref[k]);
    return v;
}

// observation gather (opf_env.py:532-549); four independent reference chains in flight per thread
template <class C>
OPFG_HD void gather_obs(const GridDev& g, const C& cx, const double* S, const OpfgBatch& B, int64_t env) {
    const int T = cx.nthreads(), n = g.n_obs;
    float* o32 = B.obs_f32 ? B.obs_f32 + env * (int64_t)n : nullptr;
    double* o64 = B.obs_f64 ? B.obs_f64 + env * (int64_t)n : nullptr;
    if (g.n_obs_runs > 0) {
        // whole columns of the state row: coalesced copies, no reference loads in front of the data loads
        for (int r = 0; r < g.n_obs_runs; ++r) {
            const int src = g.obs_runs[3 * r], dst = g.obs_runs[3 * r + 1], len = g.obs_runs[3 * r + 2];
            int k = cx.tid;
            for (; k + 3 * T < len; k += 4 * T) {          // four loads in flight per lane (the row comes from DRAM)
                const double v0 = S[src + k], v1 = S[src + k + T], v2 = S[src + k + 2 * T], v3 = S[src + k + 3 * T];
                if (o32) { o32[dst + k] = (float)v0; o32[dst + k + T] = (float)v1; o32[dst + k + 2 * T] = (float)v2; o32[dst + k + 3 * T] = (float)v3; }
                if (o64) { o64[dst + k] = v0; o64[dst + k + T] = v1; o64[dst + k + 2 * T] = v2; o64[dst + k + 3 * T] = v3; }
            }
            for (; k < len; k += T) {
                const double v = S[src + k];
                if (o32) o32[dst + k] = (float)v;
                if (o64) o64[dst + k] = v;
            }
        }
        return;
    }
    int j = cx.tid;
    for (; j + 3 * T < n; j += 4 * T) {
        const double v0 = obs_value(g, S, j), v1 = obs_value(g, S, j + T), v2 = obs_value(g, S, j + 2 * T),
                     v3 = obs_value(g, S, j + 3 * T);
        if (o32) { o32[j] = (float)v0; o32[j + T] = (float)v1; o32[j + 2 * T] = (float)v2; o32[j + 3 * T] = (float)v3; }
        if (o64) { o64[j] = v0; o64[j + T] = v1; o64[j + 2 * T] = v2; o64[j + 3 * T] = v3; }
    }
    for (; j < n; j += T) {
        const double v = obs_value(g, S, j);
        if (o32) o32[j] = (float)v;
        if (o64) o64[j] = v;
    }
}

// --------------------------------------- kernel 1b: actions -> set-points -> Sbus
template <class C>
OPFG_HD void env_assemble(const GridDev& g, const C& cx, const double* act, double* S, double* sbus,
                          double* yval_env = nullptr, double* bry_env = nullptr, bool absolute = false,
                          double* vm_out = nullptr) {
    const int T = cx.nthreads();
    for (int j = cx.tid; act != nullptr && j < g.n_act; j += T) {
        double a = act[j];
        a = a < 0.0 ? 0.0 : (a > 1.0 ? 1.0 : a);               // opf_env.py:429
        const double lo = ref_val(g, S, g.act_lo[j]), hi = ref_val(g, S, g.act_hi[j]);
        double sp = a * (hi - lo) + lo;                           // :461
        if (g.act_diff_step > 0.0 && !absolute) {                 // :451-458 incremental set-points
            const double prev = S[g.act_slot[j]] * ref_val(g, S, g.act_div[j]);
            sp = (2.0 * a - 1.0) * g.act_diff_step * (hi - lo) + prev;
            if (!g.act_clamp_lo) { if (sp > hi) sp = hi; if (sp < lo) sp = lo; }   // :464-470 (min_/max_ = lo/hi)
        }
        if (g.act_clamp_lo) {                                     // :464-470
            const double cl = ref_val(g, S, g.act_clamp_lo[j]), ch = ref_val(g, S, g.act_clamp_hi[j]);
            if (sp > ch) sp = ch;
            if (sp < cl) sp = cl;
        }
        sp /= ref_val(g, S, g.act_div[j]);                        // :472-474
        const int kind = g.act_kind[j];
        if (kind == 1) sp = (rint(sp) != 0.0) ? 1.0 : 0.0;        // :476-478
        else if (kind == 2) sp = rint(sp);                        // :479-481
        S[g.act_slot[j]] = sp;
    }
    if (sbus == nullptr) return;          // set-points only (reset applies the centre action)
    cx.sync();
#ifdef OPFG_DEVICE_BUILD
    __threadfence_block();
#endif
    if (g.n_dyn > 0 && yval_env && bry_env) {
        // kernel 1a per environment: admittances of the branches with tap / in-service cells
        // (pandapower build_branch.py tap handling + pypower makeYbus.py [ext-mem]), then Ybus values
        for (int d = cx.tid; d < g.n_dyn; d += T) {
            double p[6];
            const double* src = g.br_param + 6 * (size_t)g.dyn_branch[d];
            for (int k = 0; k < 6; ++k) p[k] = src[k];
            const int fl = g.dyn_flags[d];
            const double pos = ref_val(g, S, g.dyn_tap_ref[d]);
            if (pos == pos) {
                if (fl & OPFG_DYN_TAP_LV) {
                    // pandapower _calc_tap_from_dataframe / _calc_r_x_y_from_dataframe [ext-mem]: the LV voltage is
                    // the tapped one, so the ratio falls with t while the impedances (referred to the LV side) rise with t^2
                    const double t = 1.0 + (pos - g.dyn_neutral[d]) * g.dyn_step[d] / 100.0;
                    const double t2 = t * t * g.dyn_lv_scale[d];
                    p[4] = g.dyn_ratio0[d] / t;
                    p[0] *= t2; p[1] *= t2; p[2] /= t2; p[3] /= t2;
                } else {
                    p[4] = g.dyn_ratio0[d] * (1.0 + (pos - g.dyn_neutral[d]) * g.dyn_step[d] / 100.0);
                }
            }
            const bool cf = ref_val(g, S, g.dyn_cf_ref[d]) != 0.0, ct = ref_val(g, S, g.dyn_ct_ref[d]) != 0.0;
            bool on = ref_val(g, S, g.dyn_svc_ref[d]) != 0.0;
            on = on && ((fl & OPFG_DYN_TRAFO) ? (cf && ct) : (cf || ct));
            if (!on) { p[0] = 1e300; p[1] = 0; p[2] = 0; p[3] = 0; }
            double* y = bry_env + 8 * (size_t)d;
            branch_admittance(p, y);
            if (on && !(cf && ct)) {
                // line open at one end: pandapower hangs it from an auxiliary bus (PQ, no injection); eliminating
                // that bus leaves a shunt at the closed end: Y' = Y_cc - Y_co Y_oc / Y_oo
                const double nr = y[2] * y[4] - y[3] * y[5], ni = y[2] * y[5] + y[3] * y[4];   // Yft Ytf
                const double* o = cf ? y + 6 : y;             // Y_oo: the open end's self admittance
                const double m2 = o[0] * o[0] + o[1] * o[1];
                const double qr = (nr * o[0] + ni * o[1]) / m2, qi = (ni * o[0] - nr * o[1]) / m2;
                const double cr = (cf ? y[0] : y[6]) - qr, ci = (cf ? y[1] : y[7]) - qi;
                for (int k = 0; k < 8; ++k) y[k] = 0.0;
                y[cf ? 0 : 6] = cr; y[cf ? 1 : 7] = ci;
            }
        }
        cx.sync();
#ifdef OPFG_DEVICE_BUILD
        __threadfence_block();
#endif
        for (int e = cx.tid; e < g.nnz_y; e += T) ybus_entry(g, g.br_y, e, yval_env + 2 * (size_t)e, bry_env);
    }
    if (g.vm_from_state && vm_out) {     // start |V| / set-point of every bus (pandapower: V0[gen bus] = VG)
        bool islands = false;
        if (g.isl && bry_env) {          // is a spanning-tree branch out of service in this environment?
            double out = 0.0;
            for (int d = cx.tid; d < g.n_dyn; d += T)     // connects nothing: its Yft is zero (kernel 1a above)
                if (g.dyn_crit[d] && bry_env[8 * (size_t)d + 2] == 0.0 && bry_env[8 * (size_t)d + 3] == 0.0) out = 1.0;
            islands = cx.block_max(out) > 0.0;
        }
        for (int bus = cx.tid; bus < g.nb; bus += T) {
            const int r = g.bus_vm_ref[bus];
            const double vm = r == OPFG_NO_REF ? g.vm0_bus[bus] : ref_val(g, S, r);
            // while the walk below runs, a NEGATIVE start value means "not reached yet"; slack buses are the seeds
            vm_out[bus] = (islands && g.type_int[g.int_of_bus[bus]] != OPFG_REF) ? -vm : vm;
        }
        if (islands) {
#ifdef OPFG_DEVICE_BUILD
            volatile double* lab = vm_out;      // labels change under the readers' feet (monotonically): no caching
#else
            double* lab = vm_out;
#endif
            for (;;) {
                cx.sync();
#ifdef OPFG_DEVICE_BUILD
                __threadfence_block();
#endif
                double changed = 0.0;
                for (int bus = cx.tid; bus < g.nb; bus += T) {
                    if (lab[bus] > 0.0) continue;
                    bool hit = false;
                    for (int e = g.isl_ptr[bus]; e < g.isl_ptr[bus + 1] && !hit; ++e) {
                        const int d = g.dyn_of_branch[g.isl_br[e]];
                        if (d >= 0 && bry_env[8 * (size_t)d + 2] == 0.0 && bry_env[8 * (size_t)d + 3] == 0.0) continue;
                        hit = lab[g.isl_adj[e]] > 0.0;
                    }
                    if (hit) { lab[bus] = -lab[bus]; changed = 1.0; }
                }
                if (!(cx.block_max(changed) > 0.0)) break;
            }
            for (int bus = cx.tid; bus < g.nb; bus += T)
                if (!(lab[bus] > 0.0)) lab[bus] = 0.0;             // cut off: dropped from this power flow
        }
    }
    const double inv_base = 1.0 / g.base_mva;
    // buses in descending order of their entry count: the lanes of one round carry equal work
    for (int k = cx.tid; k < g.nb; k += T) {
        const int bus = g.inj_order[k];
        double p = 0, q = 0;
#pragma unroll 4
        for (int e = g.inj_ptr[bus]; e < g.inj_ptr[bus + 1]; ++e) {
            const double c = ref_val(g, S, g.inj_coef[e]);
            p += c * ref_val(g, S, g.inj_p[e]);
            q += c * ref_val(g, S, g.inj_q[e]);
        }
        sbus[2 * bus] = p * inv_base;
        sbus[2 * bus + 1] = q * inv_base;
    }
}

// ------------------------------------------------------ kernels 2-4: Newton-Raphson
// Shared-memory working set of one environment.  2x2 blocks are 32-byte aligned
// (two 128-bit shared loads per block); V is kept as interleaved (re, im) pairs.
// The 2x2 blocks are stored as two planes of 16-byte rows (row 0 of every block, then row 1 of
// every block): neighbouring lanes working on neighbouring blocks then touch contiguous 128-byte
// spans instead of a 32-byte stride, which halves the shared-memory bank conflicts (profile r01d).
struct PfSmem {
    double *lu, *lu1, *rhs, *vri, *ivm, *red;
    double* qadd;                 // [n] reactive power fixed at a limit (enforce_q_lims), else null
    unsigned char* type;          // [nb] per-environment bus types (enforce_q_lims), else null
    const unsigned char* bus_type;   // what the kernels read: `type` or the shared table
};

OPFG_HHD size_t pf_smem_doubles(int n_blocks, int n, int nb, int threads, int n_qlim = 0) {
    return (size_t)4 * n_blocks + 2 * (size_t)n + 3 * (size_t)nb + 2 * (size_t)(threads / 32 + 1) + 2 +
           (n_qlim > 0 ? (size_t)n + (size_t)(nb + 7) / 8 + 1 : 0);
}

OPFG_HD PfSmem pf_carve(double* base, int n_blocks, int n, int nb) {
    PfSmem s;
    s.lu = base;
    s.lu1 = base + 2 * (size_t)n_blocks;
    s.rhs = s.lu + 4 * (size_t)n_blocks;
    s.vri = s.rhs + 2 * (size_t)n;
    s.ivm = s.vri + 2 * (size_t)nb;
    s.red = s.ivm + nb + (nb & 1);
    s.qadd = nullptr; s.type = nullptr; s.bus_type = nullptr;
    return s;
}

struct D2 { double x, y; };
#ifdef OPFG_DEVICE_BUILD
OPFG_HD D2 ld2(const double* p) { const double2 v = *reinterpret_cast<const double2*>(p); return D2{v.x, v.y}; }
OPFG_HD void st2(double* p, double x, double y) { *reinterpret_cast<double2*>(p) = make_double2(x, y); }
OPFG_HD D2 ldg2(const double* p) { const double2 v = __ldg(reinterpret_cast<const double2*>(p)); return D2{v.x, v.y}; }
#else
OPFG_HD D2 ld2(const double* p) { return D2{p[0], p[1]}; }
OPFG_HD void st2(double* p, double x, double y) { p[0] = x; p[1] = y; }
OPFG_HD D2 ldg2(const double* p) { return D2{p[0], p[1]}; }
#endif

// Row part of the fused power mismatch (kernel 2) + Jacobian (kernel 3): injected
// current, S_i = V_i conj(I_i), mismatch into rhs, and -- if `jac` -- the diagonal
// 2x2 block.  Returns the row's contribution to ||F||inf.  The off-diagonal blocks
// are written entry-parallel by `jacobian_entry` (balanced over the lanes).
// Formulas: pypower dSbus_dV.py in polar form [ext-mem], SURVEY.md App. B.4.
OPFG_HD double row_mismatch(const GridDev& g, const PfSmem& s, const double* yv, const double* sbus,
                            int i, bool jac) {
    D2 sp = ldg2(sbus + 2 * g.bus_of_int[i]);                // P, Q set-point (global, issued early)
    const D2 vi = ld2(s.vri + 2 * i);
    const bool pq = s.bus_type[i] == OPFG_PQ;
    const int e0 = g.y_ptr[i], e1 = g.y_ptr[i + 1];
    double ir = 0, ii = 0, dr = 0, di = 0;
    for (int e = e0; e < e1; ++e) {
        const int j = (int)(g.y_meta[e].x & 0xffffu);
        const D2 y = ld2(yv + 2 * e);                         // table: global or staged in shared memory
        const D2 vj = ld2(s.vri + 2 * j);
        const double tr = fma(y.x, vj.x, -(y.y * vj.y)), ti = fma(y.x, vj.y, y.y * vj.x);   // Y_ij V_j
        ir += tr; ii += ti;
        if (e == e0) { dr = tr; di = ti; }                    // the diagonal entry is first
    }
    const double P = fma(vi.x, ir, vi.y * ii), Q = fma(vi.y, ir, -(vi.x * ii));   // S_i = V_i conj(I_i)
    if (g.isl && vi.x == 0.0 && vi.y == 0.0) {               // bus cut off from every slack: identity rows, no mismatch
        if (jac) { st2(s.lu + 2 * i, 1.0, 0.0); st2(s.lu1 + 2 * i, 0.0, 1.0); }
        st2(s.rhs + 2 * i, 0.0, 0.0);
        return 0.0;
    }
    if (jac) {
        const double ar = fma(vi.x, dr, vi.y * di), ai = fma(vi.y, dr, -(vi.x * di));   // V_i conj(Y_ii V_i)
        const double inv_vmi = s.ivm[i];
        st2(s.lu + 2 * i, -Q + ai, (ar + P) * inv_vmi);
        st2(s.lu1 + 2 * i, pq ? P - ar : 0.0, pq ? (ai + Q) * inv_vmi : 1.0);
    }
    if (s.qadd) sp.y += s.qadd[i];                           // first use of the set-point: its L2 latency hid behind the row
    const double dp = P - sp.x, dq = pq ? Q - sp.y : 0.0;
    st2(s.rhs + 2 * i, -dp, -dq);
    if (dp != dp || dq != dq) return NAN;
    const double a = fabs(dp), c = fabs(dq);
    return a > c ? a : c;
}

// Off-diagonal Jacobian block fed by Ybus entry e = (i, j), i != j, both non-slack.
OPFG_HD void jacobian_entry(const GridDev& g, const PfSmem& s, const double* yv, int e) {
    const U2 m = g.y_meta[e];
    const int blk = (int)(m.x >> 16) - 1;
    if (blk < 0 || blk < g.n) return;                         // ref column, or the diagonal entry
    const int j = (int)(m.x & 0xffffu), i = (int)m.y;
    const D2 y = ld2(yv + 2 * e);
    const D2 vj = ld2(s.vri + 2 * j), vi = ld2(s.vri + 2 * i);
    const double tr = fma(y.x, vj.x, -(y.y * vj.y)), ti = fma(y.x, vj.y, y.y * vj.x);
    const double ar = fma(vi.x, tr, vi.y * ti), ai = fma(vi.y, tr, -(vi.x * ti));   // V_i conj(Y_ij V_j)
    const double inv_vmj = s.ivm[j];
    const bool pq = s.bus_type[i] == OPFG_PQ;
    st2(s.lu + 2 * blk, ai, ar * inv_vmj);                    // dP/dtheta_j, dP/dVm_j
    st2(s.lu1 + 2 * blk, pq ? -ar : 0.0, pq ? ai * inv_vmj : 0.0);
}

// ---- diagonal pivot: D_k -= sum L~(k,m) W(m,k), y_k -= sum L~(k,m) t_m, invert, t_k = D^-1 y_k
// The sum runs in increasing m.  Its part over sources more than one level below k is applied
// EAGERLY, by separate items in the phases right after those source levels finish (the top of the
// elimination tree would otherwise walk its whole history in one long dependent chain while most
// lanes idle); the partial sums wait in D_k / y_k, so the order of additions -- and every bit of
// the result -- is that of the single gather.
// (all pair loops below are unrolled four times: the index and block loads of four pairs are in flight while the
// accumulators take the products IN ORDER -- the chain per pair shrinks from index -> blocks -> FMAs to the FMAs)
OPFG_HD void lu_gather_pairs(const GridDev& g, const PfSmem& s, int p, int pe, D2& r0, D2& r1, D2& y) {
#pragma unroll 4
    for (; p < pe; ++p) {
        const U2 id = g.dp_pack[p];
        const int li = 2 * (int)(id.x & 0xffffu), wi = 2 * (int)(id.x >> 16);
        const D2 l0 = ld2(s.lu + li), l1 = ld2(s.lu1 + li), w0 = ld2(s.lu + wi), w1 = ld2(s.lu1 + wi),
                 t = ld2(s.rhs + 2 * id.y);
        r0.x = fma(-l0.y, w1.x, fma(-l0.x, w0.x, r0.x));  r0.y = fma(-l0.y, w1.y, fma(-l0.x, w0.y, r0.y));
        r1.x = fma(-l1.y, w1.x, fma(-l1.x, w0.x, r1.x));  r1.y = fma(-l1.y, w1.y, fma(-l1.x, w0.y, r1.y));
        y.x = fma(-l0.y, t.y, fma(-l0.x, t.x, y.x));      y.y = fma(-l1.y, t.y, fma(-l1.x, t.x, y.y));
    }
}
OPFG_HD void lu_eager_item(const GridDev& g, const PfSmem& s, U2 it) {
    const int k = (int)(it.x & 0xffffu);
    D2 r0 = ld2(s.lu + 2 * k), r1 = ld2(s.lu1 + 2 * k), y = ld2(s.rhs + 2 * k);
    lu_gather_pairs(g, s, (int)it.y, (int)it.y + (int)(it.x >> 16), r0, r1, y);
    st2(s.lu + 2 * k, r0.x, r0.y);
    st2(s.lu1 + 2 * k, r1.x, r1.y);
    st2(s.rhs + 2 * k, y.x, y.y);
}
// one lane per pivot
OPFG_HD void lu_diag_item(const GridDev& g, const PfSmem& s, int k) {
    D2 r0 = ld2(s.lu + 2 * k), r1 = ld2(s.lu1 + 2 * k), y = ld2(s.rhs + 2 * k);
    lu_gather_pairs(g, s, g.dp_own[k], g.dp_ptr[k + 1], r0, r1, y);
    const double r = 1.0 / fma(r0.x, r1.y, -(r0.y * r1.x));
    const double ia = r1.y * r, ib = -r0.y * r, ic = -r1.x * r, id_ = r0.x * r;
    st2(s.lu + 2 * k, ia, ib);
    st2(s.lu1 + 2 * k, ic, id_);
    st2(s.rhs + 2 * k, fma(ia, y.x, ib * y.y), fma(ic, y.x, id_ * y.y));
}

// An off-diagonal item in two parts.  The GATHER (target -= sum L~ W over pairs from lower levels) depends on
// nothing its own level produces, so it runs in the same phase as the level's diagonal items -- which leave most
// lanes idle (a handful of pivots per level in the upper half of the elimination tree); the SCALE part of a U block
// (W = D_k^-1 U) waits for the barrier behind the inversion of D_k and is short.  Same operations in the same
// order as the one-piece item: same bits.
OPFG_HD void lu_off_gather(const GridDev& g, const PfSmem& s, int item) {
    const U2 hdr = g.off_hdr[item];
    const int pe = (int)(g.off_hdr[item + 1].y & 0x7fffffffu);
    int p = (int)(hdr.y & 0x7fffffffu);
    const bool fill = (hdr.y >> 31) != 0;
    if (p == pe && !fill) return;                             // a U block nothing updates: only scaled
    const int xi = 2 * (int)(hdr.x & 0xffffu);
    // a fill block (bit 31) has no stored value yet: its slot may still hold a block that died a level ago
    D2 r0{0.0, 0.0}, r1{0.0, 0.0};
    if (!fill) { r0 = ld2(s.lu + xi); r1 = ld2(s.lu1 + xi); }
#pragma unroll 4
    for (; p < pe; ++p) {
        const uint32_t id = g.op_pack[p];
        const int li = 2 * (int)(id & 0xffffu), wi = 2 * (int)(id >> 16);
        const D2 l0 = ld2(s.lu + li), l1 = ld2(s.lu1 + li), w0 = ld2(s.lu + wi), w1 = ld2(s.lu1 + wi);
        r0.x = fma(-l0.y, w1.x, fma(-l0.x, w0.x, r0.x));  r0.y = fma(-l0.y, w1.y, fma(-l0.x, w0.y, r0.y));
        r1.x = fma(-l1.y, w1.x, fma(-l1.x, w0.x, r1.x));  r1.y = fma(-l1.y, w1.y, fma(-l1.x, w0.y, r1.y));
    }
    st2(s.lu + xi, r0.x, r0.y);
    st2(s.lu1 + xi, r1.x, r1.y);
}
OPFG_HD void lu_off_scale(const GridDev& g, const PfSmem& s, int item) {
    const uint32_t hx = g.off_hdr[item].x;
    const int piv = (int)(hx >> 16) - 1;
    if (piv < 0) return;                                      // L~ blocks stay unscaled
    const int xi = 2 * (int)(hx & 0xffffu);
    const D2 r0 = ld2(s.lu + xi), r1 = ld2(s.lu1 + xi);
    const D2 i0 = ld2(s.lu + 2 * piv), i1 = ld2(s.lu1 + 2 * piv);   // W = D^-1 * U
    const double a = fma(i0.x, r0.x, i0.y * r1.x), b = fma(i0.x, r0.y, i0.y * r1.y);
    const double c = fma(i1.x, r0.x, i1.y * r1.x), d = fma(i1.x, r0.y, i1.y * r1.y);
    st2(s.lu + xi, a, b);
    st2(s.lu1 + xi, c, d);
}

OPFG_HD void bwd_item(const GridDev& g, const PfSmem& s, int k) {
    D2 x = ld2(s.rhs + 2 * k);
    const int pe = g.up_ptr[k + 1];
#pragma unroll 4
    for (int p = g.up_ptr[k]; p < pe; ++p) {
        const uint32_t id = g.up_pack[p];
        const int wi = 2 * (int)(id & 0xffffu);
        const D2 w0 = ld2(s.lu + wi), w1 = ld2(s.lu1 + wi), xj = ld2(s.rhs + 2 * (id >> 16));
        x.x = fma(-w0.y, xj.y, fma(-w0.x, xj.x, x.x));
        x.y = fma(-w1.y, xj.y, fma(-w1.x, xj.x, x.y));
    }
    st2(s.rhs + 2 * k, x.x, x.y);
}

// One environment: start values (the DC start comes from the dense pre-pass), Newton-Raphson to tolerance,
// write |V|, angle, flag.
// Mirrors pandapower newtonpf control flow (SURVEY.md App. B.4): convergence is
// tested before the first iteration; at most max_iter linear solves.
template <class C>
OPFG_HD void env_pf_solve(const GridDev& g, const C& cx, double* smem, const double* sbus,
                          const double* yval_env, double* vm_out, double* va_out,
                          uint8_t* conv_out, int32_t* iter_out) {
    const int T = cx.nthreads();
    const int n = g.n, nb = g.nb;
    PfSmem s = pf_carve(smem, g.n_blocks, n, nb);
    const double* yv = yval_env ? yval_env : g.y_val;
    OPFG_TICK_INIT;
    s.bus_type = g.type_int;
    if (g.n_qlim > 0) {   // enforce_q_lims: this environment may turn PV buses into PQ buses
        s.qadd = s.red + 2 * (T / 32 + 1) + 2;
        s.type = reinterpret_cast<unsigned char*>(s.qadd + n);
        for (int i = cx.tid; i < nb; i += T) s.type[i] = g.type_int[i];
        for (int k = cx.tid; k < n; k += T) s.qadd[k] = 0.0;
        s.bus_type = s.type;
        cx.sync();
    }

    OPFG_TICK(0);   // q-limit set-up
    // |V| and angle are touched only by their owner lane, once per iteration: they live in the
    // output buffers (L2) instead of shared memory, which buys one more resident environment per SM
    for (int i = cx.tid; i < nb; i += T) {
        const int bus = g.bus_of_int[i];
        const double vm = g.vm_from_state ? vm_out[bus] : g.vm0_int[i];
        const bool dead = g.isl && vm == 0.0;                 // kernel 1 found the bus cut off from every slack
        const double va = dead ? 0.0 : ((g.init_dc && i < n) ? va_out[bus] : g.va0_int[i]);   // DC start: written by the dense pre-pass
        double sn, cs;
        sincos(va, &sn, &cs);
        vm_out[bus] = vm; va_out[bus] = va; s.ivm[i] = dead ? 0.0 : 1.0 / vm;
        st2(s.vri + 2 * i, vm * cs, vm * sn);
    }
    cx.sync();
    OPFG_TICK(7);   // initial V

    int it = 0;
    int converged = 0;
    double prev = 1.0;
  restart_after_q_limits:
    while (true) {
        // quadratic convergence: after a norm below 1e-4 the next one is almost surely below
        // tol, so look at the mismatch alone first and build the Jacobian only if needed
        bool jac = !(prev < 1e-4);
        double nrm;
        while (true) {
            double part = 0;
            bool bad = false;
            for (int i = cx.tid; i < n; i += T) {
                const double r = row_mismatch(g, s, yv, sbus, i, jac);
                if (r != r) bad = true; else if (r > part) part = r;
            }
            if (jac) {
                for (int e = cx.tid; e < g.nnz_y_nonref; e += T) jacobian_entry(g, s, yv, e);
                // fill blocks are not zeroed here: their item starts from zero (lu_off_gather), their slot may be shared
            }
            nrm = cx.block_max(bad ? NAN : part);
            cx.sync();
            OPFG_TICK(jac ? 1 : 2);   // row pass with / without Jacobian
            if (jac || nrm < g.tol || it >= g.max_iter || nrm != nrm) break;
            jac = true;
        }
        prev = nrm;
        if (nrm < g.tol) { converged = 1; break; }
        if (it >= g.max_iter || nrm != nrm) break;
        ++it;
        for (int l = 0; l < g.n_levels; ++l) {
            const int lb = g.level_ptr[l], le = g.level_ptr[l + 1];
            const int n_own = le - lb, eb = g.eg_ptr[l], n_items = n_own + g.eg_ptr[l + 1] - eb;
            for (int idx = cx.tid; idx < n_items; idx += T) {
                if (idx < n_own) lu_diag_item(g, s, lb + idx);
                else lu_eager_item(g, s, g.eg_item[eb + idx - n_own]);
            }
            OPFG_TICK(112 + l);  // lane 0's own diagonal work (the rest of the phase: gathers of other lanes + barrier)
            // gathers of this level's off-diagonal items, from the far end of the lanes (the diagonals took the near end)
            const int ob = g.off_ptr[l], oe = g.off_ptr[l + 1];
            for (int item = ob + (T - 1 - cx.tid); item < oe; item += T) lu_off_gather(g, s, item);
            cx.sync();
            OPFG_TICK(16 + l);   // slots: 16.. diagonal (+ gather) phase, 48.. scale phase, 80.. backward (up to 32 levels)
            for (int item = ob + (T - 1 - cx.tid); item < oe; item += T) lu_off_scale(g, s, item);
            cx.sync();
            OPFG_TICK(48 + l);
        }
        for (int l = g.n_levels - 1; l >= 0; --l) {
            for (int k = g.level_ptr[l] + cx.tid; k < g.level_ptr[l + 1]; k += T) bwd_item(g, s, k);
            cx.sync();
            OPFG_TICK(80 + l);
        }
        for (int k = cx.tid; k < n; k += T) {
            const D2 dx = ld2(s.rhs + 2 * k);
            const int bus = g.bus_of_int[k];
            double va = va_out[bus] + dx.x;
            double vm = vm_out[bus] + ((s.bus_type[k] == OPFG_PQ) ? dx.y : 0.0);
            // V = Vm*exp(j*Va); Vm = |V|; Va = angle(V)  (newtonpf.py)
            if (vm < 0) { vm = -vm; va += M_PI; }
            if (va > M_PI || va <= -M_PI) va -= 2.0 * M_PI * floor((va + M_PI) / (2.0 * M_PI));
            double sn, cs;
            sincos(va, &sn, &cs);
            va_out[bus] = va; vm_out[bus] = vm; s.ivm[k] = (g.isl && vm == 0.0) ? 0.0 : 1.0 / vm;
            st2(s.vri + 2 * k, vm * cs, vm * sn);
        }
        cx.sync();
        OPFG_TICK(6);
    }
    if (converged && g.n_qlim > 0) {
        // pandapower `_run_ac_pf_with_qlims_enforced` [ext-mem]: a voltage-controlled bus whose reactive
        // output left [QMIN, QMAX] is fixed at the limit and becomes a PQ bus; solve again from the
        // current voltages until no limit is violated.
        double changed = 0;
        for (int q = cx.tid; q < g.n_qlim; q += T) {
            const int i = g.qlim_bus[q];
            if (s.type[i] != OPFG_PV) continue;
            const D2 vi = ld2(s.vri + 2 * i);
            if (g.isl && vi.x == 0.0 && vi.y == 0.0) continue;
            double ir = 0, ii = 0;
            for (int e = g.y_ptr[i]; e < g.y_ptr[i + 1]; ++e) {
                const D2 y = ld2(yv + 2 * e);
                const D2 vj = ld2(s.vri + 2 * (g.y_meta[e].x & 0xffffu));
                ir += fma(y.x, vj.x, -(y.y * vj.y));
                ii += fma(y.x, vj.y, y.y * vj.x);
            }
            const double qg = fma(vi.y, ir, -(vi.x * ii)) - sbus[2 * g.bus_of_int[i] + 1];   // generator Q, p.u.
            if (qg > g.qlim_max[q]) { s.qadd[i] = g.qlim_max[q]; s.type[i] = OPFG_PQ; changed = 1; }
            else if (qg < g.qlim_min[q]) { s.qadd[i] = g.qlim_min[q]; s.type[i] = OPFG_PQ; changed = 1; }
        }
        changed = cx.block_max(changed);
        cx.sync();
        if (changed > 0) { converged = 0; it = 0; prev = 1.0; goto restart_after_q_limits; }
    }
    if (g.isl)                         // pandapower reports NaN for the buses it dropped
        for (int k = cx.tid; k < n; k += T)
            if (s.vri[2 * k] == 0.0 && s.vri[2 * k + 1] == 0.0) {
                const int bus = g.bus_of_int[k];
                vm_out[bus] = NAN; va_out[bus] = NAN;
            }
    if (cx.tid == 0) { *conv_out = (uint8_t)converged; *iter_out = it; }
}

// ------------------------------------------- kernels 2-4, fused form for radial grids
// On a radial grid (a forest once the slack bus is removed) every pivot of a leaf-first elimination
// has ONE later neighbour, its parent: no fill, and no off-diagonal block is ever updated.  Then the
// Jacobian need not exist in memory: the thread that eliminates pivot k computes row k of the power
// mismatch, the diagonal block, the blocks L(k, child) it gathers with and the block U(k, parent) it
// scales, all from V and Ybus on the spot (the loads of V_k / V_child serve mismatch and Jacobian
// alike).  Per environment only V, 1/|V|, t and W(k, parent) live in shared memory: 8.7 KB on the
// 122-bus grid instead of 19 KB, and one phase per level instead of three plus a row pass.  The
// smaller footprint is spent on MORE, NARROWER environments per SM: T = 16 lanes per
// environment, two environments per warp, synchronised by __syncwarp alone (no block barriers).
// Every sum runs in the order of env_pf_solve: same bits.
struct TreeSmem { double *vri, *ivm, *t, *w0, *w1; };
OPFG_HHD size_t tree_smem_doubles(int n, int nb) {
    size_t d = 2 * (size_t)nb + (size_t)(nb + (nb & 1)) + 6 * (size_t)n + (n & 1) * 2;
    while (d % 16 != 4) d += 2;          // environment stride = 32 B mod 128 B: neighbours start in other banks
    return d;
}
OPFG_HD TreeSmem tree_carve(double* base, int n, int nb) {
    TreeSmem s;
    s.vri = base; s.ivm = s.vri + 2 * (size_t)nb; s.t = s.ivm + nb + (nb & 1);
    s.w0 = s.t + 2 * (size_t)n; s.w1 = s.w0 + 2 * (size_t)n;
    return s;
}

#ifdef OPFG_DEVICE_BUILD
template <int T>
struct Grp {
    static constexpr int OWN_ROUNDS = 128 / T;
    int tid;                                   // lane within the environment's group of T lanes
    __device__ __forceinline__ int nthreads() const { return T; }
    __device__ __forceinline__ void sync() const { __syncwarp(); }
    __device__ __forceinline__ bool any(bool p) const { return __any_sync(0xffffffffu, p) != 0; }
    __device__ __forceinline__ double group_max(double v) const {   // NaN-propagating, over the T lanes
        double bad = (v != v) ? 1.0 : 0.0;
        v = bad > 0 ? 0.0 : v;
#pragma unroll
        for (int o = T / 2; o > 0; o >>= 1) {
            v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
            bad = fmax(bad, __shfl_xor_sync(0xffffffffu, bad, o));
        }
        return bad > 0 ? NAN : v;
    }
};
#else
template <int T>
struct Grp {
    static constexpr int OWN_ROUNDS = 8;
    int tid = 0;
    int nthreads() const { return 1; }
    void sync() const {}
    bool any(bool p) const { return p; }
    double group_max(double v) const { return v; }
};
#endif

// Pivot k in ONE pass over its Ybus row: every entry feeds the row's injected current (power mismatch,
// returned as the row's share of ||F||inf); if JAC, a child entry (an earlier pivot) also yields the
// block L(k, child), which is multiplied with the child's W and t right away, and the parent entry is
// remembered for U(k, parent).  After the pass: D_k = J_kk - sum L W, y_k = -F_k - sum L t, t_k = D_k^-1 y_k,
// W_k = D_k^-1 U(k, parent).  (The sums are formed before they are subtracted from J_kk, so the last bits
// differ from env_pf_solve, which subtracts product by product.)
struct TreeAcc {
    double ir, ii, g00, g01, g10, g11, gy0, gy1, ptr, pti;
    int pj;
};
// one off-diagonal Ybus entry (k, j) of pivot k, its values already loaded
template <bool JAC>
OPFG_HD void tree_entry(const TreeSmem& s, TreeAcc& a, uint32_t ent, D2 y, D2 vj, D2 vk, bool pq) {
    const double tr = fma(y.x, vj.x, -(y.y * vj.y)), ti = fma(y.x, vj.y, y.y * vj.x);   // Y_kj V_j
    a.ir += tr; a.ii += ti;
    if (JAC) {
        const uint32_t kind = ent >> 16;
        if (kind == 1u) {                                     // child: L(k, j) times the child's W and t
            const int j = (int)(ent & 0xffffu);
            const double ar = fma(vk.x, tr, vk.y * ti), ai = fma(vk.y, tr, -(vk.x * ti));   // V_k conj(Y_kj V_j)
            const double inv_vmj = s.ivm[j];
            const double l00 = ai, l01 = ar * inv_vmj, l10 = pq ? -ar : 0.0, l11 = pq ? ai * inv_vmj : 0.0;
            const D2 w0 = ld2(s.w0 + 2 * j), w1 = ld2(s.w1 + 2 * j), t = ld2(s.t + 2 * j);
            a.g00 = fma(l01, w1.x, fma(l00, w0.x, a.g00));  a.g01 = fma(l01, w1.y, fma(l00, w0.y, a.g01));
            a.g10 = fma(l11, w1.x, fma(l10, w0.x, a.g10));  a.g11 = fma(l11, w1.y, fma(l10, w0.y, a.g11));
            a.gy0 = fma(l01, t.y, fma(l00, t.x, a.gy0));    a.gy1 = fma(l11, t.y, fma(l10, t.x, a.gy1));
        } else if (kind == 2u) { a.ptr = tr; a.pti = ti; a.pj = (int)(ent & 0xffffu); }
    }
}

template <bool JAC, bool ISL = false>
OPFG_HD double tree_row(const GridDev& g, const TreeSmem& s, const double* yv, D2 sp, int k) {
    const D2 vk = ld2(s.vri + 2 * k);
    const bool dead = ISL && vk.x == 0.0 && vk.y == 0.0;      // cut off from every slack (kernel 1): V stays 0
    const bool pq = g.tr_type[k] == OPFG_PQ;
    const int e0 = g.tr_y_ptr[k], e1 = g.tr_y_ptr[k + 1];
    TreeAcc a{0, 0, 0, 0, 0, 0, 0, 0, 0, 0, -1};
    double dr, di;
    {                                                         // the diagonal entry is first
        const D2 y = ld2(yv + 2 * e0);
        dr = fma(y.x, vk.x, -(y.y * vk.y)); di = fma(y.x, vk.y, y.y * vk.x);
        a.ir = dr; a.ii = di;
    }
    int e = e0 + 1;
    // two entries per trip: their loads overlap.  (Measured alternative: ONE entry per trip with the next entry's
    // operands requested a trip ahead -- a single copy of the child / parent code per warp -- is 4 % slower.)
    for (; e + 1 < e1; e += 2) {
        const uint32_t ea = g.tr_y_ent[e], eb = g.tr_y_ent[e + 1];
        const D2 ya = ld2(yv + 2 * e), yb = ld2(yv + 2 * e + 2);
        const D2 va = ld2(s.vri + 2 * (ea & 0xffffu)), vb = ld2(s.vri + 2 * (eb & 0xffffu));
        tree_entry<JAC>(s, a, ea, ya, va, vk, pq);
        tree_entry<JAC>(s, a, eb, yb, vb, vk, pq);
    }
    if (e < e1) {
        const uint32_t ea = g.tr_y_ent[e];
        tree_entry<JAC>(s, a, ea, ld2(yv + 2 * e), ld2(s.vri + 2 * (ea & 0xffffu)), vk, pq);
    }
    const double P = fma(vk.x, a.ir, vk.y * a.ii), Q = fma(vk.y, a.ir, -(vk.x * a.ii));   // S_k = V_k conj(I_k)
    const double dp = dead ? 0.0 : P - sp.x, dq = (pq && !dead) ? Q - sp.y : 0.0;
    double res;
    if (dp != dp || dq != dq) res = NAN;
    else { const double x = fabs(dp), c = fabs(dq); res = x > c ? x : c; }
    if (!JAC) return res;
    const double ar = fma(vk.x, dr, vk.y * di), ai = fma(vk.y, dr, -(vk.x * di));   // V_k conj(Y_kk V_k)
    const double inv_vmk = s.ivm[k];
    const double d00 = dead ? 1.0 : (-Q + ai) - a.g00, d01 = (ar + P) * inv_vmk - a.g01;
    const double d10 = (pq ? P - ar : 0.0) - a.g10, d11 = dead ? 1.0 : (pq ? (ai + Q) * inv_vmk : 1.0) - a.g11;
    const double y0 = -dp - a.gy0, y1 = -dq - a.gy1;
    const double r = 1.0 / fma(d00, d11, -(d01 * d10));
    const double ia = d11 * r, ib = -d01 * r, ic = -d10 * r, id_ = d00 * r;
    st2(s.t + 2 * k, fma(ia, y0, ib * y1), fma(ic, y0, id_ * y1));
    if (a.pj >= 0) {                                          // U(k, parent) -> W_k
        const double ur = fma(vk.x, a.ptr, vk.y * a.pti), ui = fma(vk.y, a.ptr, -(vk.x * a.pti));
        const double inv_vmj = s.ivm[a.pj];
        const double u00 = ui, u01 = ur * inv_vmj, u10 = pq ? -ur : 0.0, u11 = pq ? ui * inv_vmj : 0.0;
        st2(s.w0 + 2 * k, fma(ia, u00, ib * u10), fma(ia, u01, ib * u11));
        st2(s.w1 + 2 * k, fma(ic, u00, id_ * u10), fma(ic, u01, id_ * u11));
    }
    return res;
}

template <class C, bool ISL_T = false>
OPFG_HD void env_pf_tree(const GridDev& g, const C& cx, double* smem, const double* sbus, const double* yval_env,
                         double* vm_out, double* va_out, uint8_t* conv_out, int32_t* iter_out, bool live) {
    const int T = cx.nthreads();
    const int n = g.n, nb = g.nb;
    const TreeSmem s = tree_carve(smem, n, nb);
    const double* yv = yval_env ? yval_env : g.tr_y_val;
    // |V| and angle of the buses a lane owns (bus tid + r T) stay in ITS REGISTERS for the whole solve:
    // the polar update then needs no round trip to the output buffers in L2 (11 % of the kernel's stall
    // samples before).  Buses beyond OWN rounds (large grids) keep using the output buffers.
    constexpr int OWN = C::OWN_ROUNDS;       // 128 / T on the device: grids up to 128 buses stay in registers
    double vm_own[OWN], va_own[OWN];
#pragma unroll
    for (int r = 0; r < OWN; ++r) {
        const int i = cx.tid + r * T;
        vm_own[r] = va_own[r] = 0.0;
        if (i < nb) {
            const int bus = g.tr_bus_of_int[i];
            const double vm = g.vm_from_state ? vm_out[bus] : g.tr_vm0[i];
            const bool dead = ISL_T && g.isl && vm == 0.0;      // kernel 1 found the bus cut off from every slack
            const double va = dead ? 0.0 : ((g.init_dc && i < n) ? va_out[bus] : g.tr_va0[i]);   // DC start: written by the dense pre-pass
            double sn, cs;
            sincos(va, &sn, &cs);
            vm_own[r] = vm; va_own[r] = va;
            s.ivm[i] = dead ? 0.0 : 1.0 / vm;
            st2(s.vri + 2 * i, vm * cs, vm * sn);
        }
    }
    for (int i = cx.tid + OWN * T; i < nb; i += T) {
        const int bus = g.tr_bus_of_int[i];
        const double vm = g.vm_from_state ? vm_out[bus] : g.tr_vm0[i];
        const bool dead = ISL_T && g.isl && vm == 0.0;
        const double va = dead ? 0.0 : ((g.init_dc && i < n) ? va_out[bus] : g.tr_va0[i]);
        double sn, cs;
        sincos(va, &sn, &cs);
        if (live) { vm_out[bus] = vm; va_out[bus] = va; }
        s.ivm[i] = dead ? 0.0 : 1.0 / vm;
        st2(s.vri + 2 * i, vm * cs, vm * sn);
    }
    cx.sync();
    bool active = live;
    int it = 0, converged = 0;
    double prev = 1.0;
    while (cx.any(active)) {
        if (!cx.any(active && !(prev < 1e-4))) {
            // every environment of the warp that still runs expects to have converged: mismatch alone
            double part = 0;
            bool bad = false;
            for (int k = cx.tid; k < n; k += T) {
                const double r = tree_row<false, ISL_T>(g, s, yv, ldg2(sbus + 2 * g.tr_bus_of_int[k]), k);
                if (r != r) bad = true; else if (r > part) part = r;
            }
            const double nrm = cx.group_max(bad ? NAN : part);
            if (active) {
                prev = nrm;
                if (nrm < g.tol) { converged = 1; active = false; }
                else if (it >= g.max_iter || nrm != nrm) active = false;
            }
            if (!cx.any(active)) break;
        }
        double part = 0;
        bool bad = false;
        // leaves first, one phase per level; the set-point of the NEXT level's pivot (global memory) is
        // requested before this level's pivot is worked on
        D2 sp_next{0, 0};
        { const int k0 = g.tr_level_ptr[0] + cx.tid; if (k0 < g.tr_level_ptr[1]) sp_next = ldg2(sbus + 2 * g.tr_bus_of_int[k0]); }
        for (int l = 0; l < g.n_levels; ++l) {
            const int le = g.tr_level_ptr[l + 1];
            const D2 sp0 = sp_next;
            if (l + 1 < g.n_levels) {
                const int k1 = le + cx.tid;
                if (k1 < g.tr_level_ptr[l + 2]) sp_next = ldg2(sbus + 2 * g.tr_bus_of_int[k1]);
            }
            int k = g.tr_level_ptr[l] + cx.tid;
            if (k < le) {
                double r = tree_row<true, ISL_T>(g, s, yv, sp0, k);
                if (r != r) bad = true; else if (r > part) part = r;
                for (k += T; k < le; k += T) {                // levels wider than the group (unbalanced schedule)
                    r = tree_row<true, ISL_T>(g, s, yv, ldg2(sbus + 2 * g.tr_bus_of_int[k]), k);
                    if (r != r) bad = true; else if (r > part) part = r;
                }
            }
            cx.sync();
        }
        const double nrm = cx.group_max(bad ? NAN : part);
        bool step = false;
        if (active) {
            prev = nrm;
            if (nrm < g.tol) { converged = 1; active = false; }
            else if (it >= g.max_iter || nrm != nrm) active = false;
            else { ++it; step = true; }
        }
        if (!cx.any(step)) continue;
        for (int l = g.n_levels - 1; l >= 0; --l) {           // x_k = t_k - W_k x_parent
            const int le = g.tr_level_ptr[l + 1];
            for (int k = g.tr_level_ptr[l] + cx.tid; k < le; k += T) {
                const int p = g.tr_parent[k];
                if (p < 0) continue;
                D2 x = ld2(s.t + 2 * k);
                const D2 w0 = ld2(s.w0 + 2 * k), w1 = ld2(s.w1 + 2 * k), xj = ld2(s.t + 2 * p);
                x.x = fma(-w0.y, xj.y, fma(-w0.x, xj.x, x.x));
                x.y = fma(-w1.y, xj.y, fma(-w1.x, xj.x, x.y));
                st2(s.t + 2 * k, x.x, x.y);
            }
            cx.sync();
        }
        if (step) {                                              // polar update (newtonpf.py)
#pragma unroll
            for (int r = 0; r < OWN; ++r) {
                const int k = cx.tid + r * T;
                if (k < n) {
                    const D2 dx = ld2(s.t + 2 * k);
                    double va = va_own[r] + dx.x;
                    double vm = vm_own[r] + ((g.tr_type[k] == OPFG_PQ) ? dx.y : 0.0);
                    if (vm < 0) { vm = -vm; va += M_PI; }
                    if (va > M_PI || va <= -M_PI) va -= 2.0 * M_PI * floor((va + M_PI) / (2.0 * M_PI));
                    double sn, cs;
                    sincos(va, &sn, &cs);
                    va_own[r] = va; vm_own[r] = vm; s.ivm[k] = (ISL_T && vm == 0.0) ? 0.0 : 1.0 / vm;
                    st2(s.vri + 2 * k, vm * cs, vm * sn);
                }
            }
            for (int k = cx.tid + OWN * T; k < n; k += T) {
                const D2 dx = ld2(s.t + 2 * k);
                const int bus = g.tr_bus_of_int[k];
                double va = va_out[bus] + dx.x;
                double vm = vm_out[bus] + ((g.tr_type[k] == OPFG_PQ) ? dx.y : 0.0);
                if (vm < 0) { vm = -vm; va += M_PI; }
                if (va > M_PI || va <= -M_PI) va -= 2.0 * M_PI * floor((va + M_PI) / (2.0 * M_PI));
                double sn, cs;
                sincos(va, &sn, &cs);
                va_out[bus] = va; vm_out[bus] = vm; s.ivm[k] = (ISL_T && vm == 0.0) ? 0.0 : 1.0 / vm;
                st2(s.vri + 2 * k, vm * cs, vm * sn);
            }
        }
        cx.sync();
    }
    if (live) {
#pragma unroll
        for (int r = 0; r < OWN; ++r) {
            const int i = cx.tid + r * T;
            if (i < nb) {
                const int bus = g.tr_bus_of_int[i];
                const bool dead = ISL_T && g.isl && vm_own[r] == 0.0;   // pandapower reports NaN for the buses it dropped
                vm_out[bus] = dead ? NAN : vm_own[r]; va_out[bus] = dead ? NAN : va_own[r];
            }
        }
        if (ISL_T && g.isl)
            for (int i = cx.tid + OWN * T; i < nb; i += T) {
                const int bus = g.tr_bus_of_int[i];
                if (vm_out[bus] == 0.0) { vm_out[bus] = NAN; va_out[bus] = NAN; }
            }
    }
    if (live && cx.tid == 0) { *conv_out = (uint8_t)converged; *iter_out = it; }
}

// ------------------------------------------- kernels 2-4, lane-per-environment form
// One LANE per environment: a warp walks the row-wise schedule once for 32 environments.  Every
// index is warp-uniform (no per-lane index loads, no divergence, no barriers, no shuffles), every
// per-environment value lives at [slot][lane] (coalesced / bank-conflict free).  The Jacobian is never
// stored: row k is rebuilt in a small row buffer (shared memory) from V and Ybus at the moment it is
// eliminated, and only W(k, j) = D_k^-1 U(k, j) and t_k = D_k^-1 y_k leave it, into a per-warp scratch
// area in global memory that the backward substitution reads back (L2).  All sums run in the order of
// the CTA-per-environment kernel above: both produce the same bits.
template <int LANES>
struct LaneMem {
    double *vr, *vi, *vm, *va, *ivm;   // [nb] per lane
    double *sp, *sq;                   // [n]  bus injection (set-point), internal order
    double *t;                         // [2 n]
    double *w;                         // [4 n_up]
    double *rb;                        // [4 max_row] row buffer
    double *qadd, *pqf;                // [n] enforce_q_lims: reactive power fixed at a limit; 1.0 = PQ bus
    double *yv;                        // [2 nnz_y_nonref] per-environment Ybus values (tap / in-service cells)
};
OPFG_HHD size_t lane_scratch_doubles(int nb, int n, int n_up, int nnz_nonref) {
    return 5 * (size_t)nb + 6 * (size_t)n + 4 * (size_t)n_up + 2 * (size_t)nnz_nonref;
}
template <int LANES>
OPFG_HD LaneMem<LANES> lane_carve(double* base, double* rb, int nb, int n, int n_up) {
    LaneMem<LANES> s;
    s.vr = base; s.vi = s.vr + (size_t)nb * LANES; s.vm = s.vi + (size_t)nb * LANES;
    s.va = s.vm + (size_t)nb * LANES; s.ivm = s.va + (size_t)nb * LANES;
    s.sp = s.ivm + (size_t)nb * LANES; s.sq = s.sp + (size_t)n * LANES;
    s.t = s.sq + (size_t)n * LANES; s.w = s.t + 2 * (size_t)n * LANES;
    s.qadd = s.w + 4 * (size_t)n_up * LANES; s.pqf = s.qadd + (size_t)n * LANES;
    s.yv = s.pqf + (size_t)n * LANES;
    s.rb = rb;
    return s;
}
#define OPFG_LN(p, i) (p)[(size_t)(i) * LANES]

#ifdef OPFG_DEVICE_BUILD
OPFG_HD bool lanes_any(bool p) { return __any_sync(0xffffffffu, p) != 0; }
#else
OPFG_HD bool lanes_any(bool p) { return p; }
#endif

// Rows 0..n-1 in elimination order: power mismatch of the row (-> ||F||inf of this lane's environment)
// and, if JAC, the row of the Jacobian, its elimination against the earlier rows, t_k and W(k, .).
template <int LANES, bool JAC, bool QLIM, bool DYN>
OPFG_HD double lanes_rows(const GridDev& g, const LaneMem<LANES>& s) {
    const int n = g.n;
    double part = 0.0;
    bool bad = false;
    for (int k = 0; k < n; ++k) {
        const int* hdr = g.ln_row + 4 * k;
        const int e0 = hdr[0], e1 = hdr[4];
        const double vkr = OPFG_LN(s.vr, k), vki = OPFG_LN(s.vi, k);
        const bool pq = QLIM ? OPFG_LN(s.pqf, k) != 0.0 : g.ln_type[k] == OPFG_PQ;
        double ir = 0, ii = 0, dr = 0, di = 0;
        for (int e = e0; e < e1; ++e) {
            const uint32_t meta = g.ln_y[e];
            const int j = (int)(meta & 0xffffu);
            const double yr = DYN ? OPFG_LN(s.yv, 2 * e) : g.ln_yval[2 * e];
            const double yi = DYN ? OPFG_LN(s.yv, 2 * e + 1) : g.ln_yval[2 * e + 1];
            const double vjr = OPFG_LN(s.vr, j), vji = OPFG_LN(s.vi, j);
            const double tr = fma(yr, vjr, -(yi * vji)), ti = fma(yr, vji, yi * vjr);   // Y_kj V_j
            ir += tr; ii += ti;
            if (e == e0) { dr = tr; di = ti; }                // the diagonal entry is first
            else if (JAC) {
                const int rp = (int)(meta >> 16) - 1;
                if (rp >= 0) {                                // off-diagonal block (k, j), j not a slack bus
                    const double ar = fma(vkr, tr, vki * ti), ai = fma(vki, tr, -(vkr * ti));   // V_k conj(Y_kj V_j)
                    const double inv_vmj = OPFG_LN(s.ivm, j);
                    double* b = s.rb + (size_t)(4 * rp) * LANES;
                    b[0] = ai; b[LANES] = ar * inv_vmj;
                    b[2 * LANES] = pq ? -ar : 0.0; b[3 * LANES] = pq ? ai * inv_vmj : 0.0;
                }
            }
        }
        const double P = fma(vkr, ir, vki * ii), Q = fma(vki, ir, -(vkr * ii));   // S_k = V_k conj(I_k)
        double sq = OPFG_LN(s.sq, k);
        if (QLIM) sq += OPFG_LN(s.qadd, k);
        const double dp = P - OPFG_LN(s.sp, k), dq = pq ? Q - sq : 0.0;
        if (dp != dp || dq != dq) bad = true;
        else { const double a = fabs(dp), c = fabs(dq), r = a > c ? a : c; if (r > part) part = r; }
        if (!JAC) continue;
        // diagonal block and right-hand side of the row
        double d00, d01, d10, d11, y0 = -dp, y1 = -dq;
        {
            const double ar = fma(vkr, dr, vki * di), ai = fma(vki, dr, -(vkr * di));   // V_k conj(Y_kk V_k)
            const double inv_vmk = OPFG_LN(s.ivm, k);
            d00 = -Q + ai; d01 = (ar + P) * inv_vmk;
            d10 = pq ? P - ar : 0.0; d11 = pq ? (ai + Q) * inv_vmk : 1.0;
        }
        const int dpos = g.ln_diag_pos[k];
        for (int f = hdr[1]; f < hdr[5]; ++f) {
            double* b = s.rb + (size_t)(4 * g.ln_fill[f]) * LANES;
            b[0] = 0.0; b[LANES] = 0.0; b[2 * LANES] = 0.0; b[3 * LANES] = 0.0;
        }
        // eliminate the earlier rows m (increasing): row_k -= L(k, m) W(m, .), y_k -= L(k, m) t_m
        for (int it = hdr[2]; it < hdr[6]; ++it) {
            const uint32_t el = g.ln_el[it];
            const double* lb = s.rb + (size_t)(4 * (el & 0xffffu)) * LANES;
            const double l00 = lb[0], l01 = lb[LANES], l10 = lb[2 * LANES], l11 = lb[3 * LANES];
            const int m = (int)(el >> 16);
            const double t0 = OPFG_LN(s.t, 2 * m), t1 = OPFG_LN(s.t, 2 * m + 1);
            y0 = fma(-l01, t1, fma(-l00, t0, y0));
            y1 = fma(-l11, t1, fma(-l10, t0, y1));
            for (int u = g.ln_el_uptr[it]; u < g.ln_el_uptr[it + 1]; ++u) {
                const uint32_t up = g.ln_upd[u];
                const double* wb = s.w + (size_t)(4 * (up & 0xffffu)) * LANES;
                const double w00 = wb[0], w01 = wb[LANES], w10 = wb[2 * LANES], w11 = wb[3 * LANES];
                const int tp = (int)(up >> 16);
                if (tp == dpos) {
                    d00 = fma(-l01, w10, fma(-l00, w00, d00)); d01 = fma(-l01, w11, fma(-l00, w01, d01));
                    d10 = fma(-l11, w10, fma(-l10, w00, d10)); d11 = fma(-l11, w11, fma(-l10, w01, d11));
                } else {
                    double* b = s.rb + (size_t)(4 * tp) * LANES;
                    b[0] = fma(-l01, w10, fma(-l00, w00, b[0]));
                    b[LANES] = fma(-l01, w11, fma(-l00, w01, b[LANES]));
                    b[2 * LANES] = fma(-l11, w10, fma(-l10, w00, b[2 * LANES]));
                    b[3 * LANES] = fma(-l11, w11, fma(-l10, w01, b[3 * LANES]));
                }
            }
        }
        // D_k^-1, t_k = D_k^-1 y_k, W(k, j) = D_k^-1 U(k, j)
        const double r = 1.0 / fma(d00, d11, -(d01 * d10));
        const double ia = d11 * r, ib = -d01 * r, ic = -d10 * r, id_ = d00 * r;
        OPFG_LN(s.t, 2 * k) = fma(ia, y0, ib * y1);
        OPFG_LN(s.t, 2 * k + 1) = fma(ic, y0, id_ * y1);
        for (int p = hdr[3]; p < hdr[7]; ++p) {
            const double* ub = s.rb + (size_t)(4 * (g.ln_up[p] >> 16)) * LANES;
            const double u00 = ub[0], u01 = ub[LANES], u10 = ub[2 * LANES], u11 = ub[3 * LANES];
            double* wb = s.w + (size_t)(4 * p) * LANES;
            wb[0] = fma(ia, u00, ib * u10); wb[LANES] = fma(ia, u01, ib * u11);
            wb[2 * LANES] = fma(ic, u00, id_ * u10); wb[3 * LANES] = fma(ic, u01, id_ * u11);
        }
    }
    return bad ? NAN : part;
}

// One environment per lane: start values, Newton-Raphson to tolerance, |V|, angle, flag.  Same control
// flow per environment as env_pf_solve (pandapower newtonpf, SURVEY.md App. B.4); which pass a WARP runs
// next (mismatch only, or mismatch + factorisation) is decided by vote and does not change any lane's result.
template <int LANES, bool QLIM, bool DYN>
OPFG_HD void lanes_pf_solve(const GridDev& g, const LaneMem<LANES>& s, const double* sbus, const double* yval,
                            double* vm_out, double* va_out, uint8_t* conv_out, int32_t* iter_out, bool live) {
    const int n = g.n, nb = g.nb;
    for (int i = 0; i < nb; ++i) {
        const int bus = g.ln_bus_of_int[i];
        const double vm = g.vm_from_state ? vm_out[bus] : g.ln_vm0[i];
        const double va = (g.init_dc && i < n) ? va_out[bus] : g.ln_va0[i];   // DC start: written by the dense pre-pass
        double sn, cs;
        sincos(va, &sn, &cs);
        OPFG_LN(s.vm, i) = vm; OPFG_LN(s.va, i) = va; OPFG_LN(s.ivm, i) = 1.0 / vm;
        OPFG_LN(s.vr, i) = vm * cs; OPFG_LN(s.vi, i) = vm * sn;
        if (i < n) {
            OPFG_LN(s.sp, i) = sbus[2 * bus]; OPFG_LN(s.sq, i) = sbus[2 * bus + 1];
            if (QLIM) { OPFG_LN(s.qadd, i) = 0.0; OPFG_LN(s.pqf, i) = g.ln_type[i] == OPFG_PQ ? 1.0 : 0.0; }
        }
    }
    if (DYN)
        for (int e = 0; e < 2 * g.nnz_y_nonref; ++e) OPFG_LN(s.yv, e) = yval[e];
    bool active = live;
    int it = 0, converged = 0;
    double prev = 1.0;
    for (;;) {
        while (lanes_any(active)) {
            if (!lanes_any(active && !(prev < 1e-4))) {
                // every environment still running expects to have converged: look at the mismatch alone
                const double nrm = lanes_rows<LANES, false, QLIM, DYN>(g, s);
                if (active) {
                    prev = nrm;
                    if (nrm < g.tol) { converged = 1; active = false; }
                    else if (it >= g.max_iter || nrm != nrm) active = false;
                }
                if (!lanes_any(active)) break;
            }
            const double nrm = lanes_rows<LANES, true, QLIM, DYN>(g, s);
            bool step = false;
            if (active) {
                prev = nrm;
                if (nrm < g.tol) { converged = 1; active = false; }
                else if (it >= g.max_iter || nrm != nrm) active = false;
                else { ++it; step = true; }
            }
            if (!lanes_any(step)) continue;
            for (int k = n - 1; k >= 0; --k) {                       // backward substitution
                double x0 = OPFG_LN(s.t, 2 * k), x1 = OPFG_LN(s.t, 2 * k + 1);
                const int pe = g.ln_row[4 * k + 7];
                for (int p = g.ln_row[4 * k + 3]; p < pe; ++p) {
                    const double* wb = s.w + (size_t)(4 * p) * LANES;
                    const int j = (int)(g.ln_up[p] & 0xffffu);
                    const double xj0 = OPFG_LN(s.t, 2 * j), xj1 = OPFG_LN(s.t, 2 * j + 1);
                    x0 = fma(-wb[LANES], xj1, fma(-wb[0], xj0, x0));
                    x1 = fma(-wb[3 * LANES], xj1, fma(-wb[2 * LANES], xj0, x1));
                }
                OPFG_LN(s.t, 2 * k) = x0; OPFG_LN(s.t, 2 * k + 1) = x1;
            }
            for (int k = 0; k < n; ++k) {                            // polar update (newtonpf.py)
                if (!step) continue;
                const bool pq = QLIM ? OPFG_LN(s.pqf, k) != 0.0 : g.ln_type[k] == OPFG_PQ;
                double va = OPFG_LN(s.va, k) + OPFG_LN(s.t, 2 * k);
                double vm = OPFG_LN(s.vm, k) + (pq ? OPFG_LN(s.t, 2 * k + 1) : 0.0);
                if (vm < 0) { vm = -vm; va += M_PI; }
                if (va > M_PI || va <= -M_PI) va -= 2.0 * M_PI * floor((va + M_PI) / (2.0 * M_PI));
                double sn, cs;
                sincos(va, &sn, &cs);
                OPFG_LN(s.va, k) = va; OPFG_LN(s.vm, k) = vm; OPFG_LN(s.ivm, k) = 1.0 / vm;
                OPFG_LN(s.vr, k) = vm * cs; OPFG_LN(s.vi, k) = vm * sn;
            }
        }
        if (!QLIM) break;
        // pandapower `_run_ac_pf_with_qlims_enforced` [ext-mem], as in env_pf_solve: a voltage-controlled bus
        // whose reactive output left [QMIN, QMAX] is fixed at the limit, becomes a PQ bus, solve again
        bool changed = false;
        for (int q = 0; q < g.n_qlim; ++q) {
            const int i = g.ln_qbus[q];
            const double vkr = OPFG_LN(s.vr, i), vki = OPFG_LN(s.vi, i);
            double ir = 0, ii = 0;
            for (int e = g.ln_row[4 * i]; e < g.ln_row[4 * i + 4]; ++e) {
                const int j = (int)(g.ln_y[e] & 0xffffu);
                const double yr = DYN ? OPFG_LN(s.yv, 2 * e) : g.ln_yval[2 * e];
                const double yi = DYN ? OPFG_LN(s.yv, 2 * e + 1) : g.ln_yval[2 * e + 1];
                const double vjr = OPFG_LN(s.vr, j), vji = OPFG_LN(s.vi, j);
                ir += fma(yr, vjr, -(yi * vji));
                ii += fma(yr, vji, yi * vjr);
            }
            const double qg = fma(vki, ir, -(vkr * ii)) - OPFG_LN(s.sq, i);   // generator Q, p.u.
            if (converged && OPFG_LN(s.pqf, i) == 0.0) {
                if (qg > g.ln_qmax[q]) { OPFG_LN(s.qadd, i) = g.ln_qmax[q]; OPFG_LN(s.pqf, i) = 1.0; changed = true; }
                else if (qg < g.ln_qmin[q]) { OPFG_LN(s.qadd, i) = g.ln_qmin[q]; OPFG_LN(s.pqf, i) = 1.0; changed = true; }
            }
        }
        if (changed) { converged = 0; it = 0; prev = 1.0; active = true; }
        if (!lanes_any(active)) break;
    }
    if (live) {
        for (int i = 0; i < nb; ++i) {
            const int bus = g.ln_bus_of_int[i];
            vm_out[bus] = OPFG_LN(s.vm, i); va_out[bus] = OPFG_LN(s.va, i);
        }
        *conv_out = (uint8_t)converged; *iter_out = it;
    }
}

// ------------------------------------------------------------- kernel 5: scoring
struct ScoreSmem {
    double *vr, *vi, *vm, *red;
};

OPFG_HHD size_t score_smem_doubles(int nb, int nbr, int threads) {
    (void)nbr;
    return 3 * (size_t)nb + (nb & 1) + 2 * (size_t)(threads / 32 + 1);
}

OPFG_HD double pwl_cost(const GridDev& g, const double* S, int row, double v) {
    // opfgym/objective.py:57-77; `beyond` has no sign test (SURVEY.md A.6 quirk 4)
    const double sg = (v > 0) - (v < 0);
    const double mag = fabs(v);
    double total = 0;
    for (int k = 0; k < g.n_pwl_seg; ++k) {
        const int* r = g.pwl_seg + 3 * ((size_t)row * g.n_pwl_seg + k);
        const double lo = ref_val(g, S, r[0]), hi = ref_val(g, S, r[1]), price = ref_val(g, S, r[2]);
        const double alo = fabs(lo), ahi = fabs(hi);
        const double near_ = alo < ahi ? alo : ahi, far_ = alo < ahi ? ahi : alo;
        const double ssum = lo + hi;
        const double sref = (ssum > 0) - (ssum < 0);
        const bool beyond = mag > far_;
        const bool within = (mag > near_) && (sg == sref) && !beyond && (v == v);
        if (beyond) total += sg * (hi - lo) * price;
        if (within) total += sg * (mag - near_) * price;
    }
    return total;
}

template <class C>
OPFG_HD void env_score(const GridDev& g, const C& cx, double* smem, const OpfgBatch& B, int64_t env,
                       const double* yval_env, double* S) {
    double* const stats = B.stats ? B.stats + (B.stats_slots > 1 ? (size_t)((uint64_t)env % (uint32_t)B.stats_slots) * OPFG_N_STATS : 0) : nullptr;
    const int T = cx.nthreads();
    const int nb = g.nb, nbr = g.nbr, nc = g.n_con;
    ScoreSmem s;
    s.vr = smem; s.vi = s.vr + nb; s.vm = s.vi + nb;
    s.red = s.vm + nb + (nb & 1);
    // S: this environment's state row -- in global memory, or a shared-memory copy staged by the caller
    const double* vm = B.vm + env * (int64_t)nb;
    const double* va = B.va + env * (int64_t)nb;
    const double* sbus = B.sbus + env * (int64_t)nb * 2;
#ifdef OPFG_DEVICE_BUILD
    // (issued before the converged flag is looked at: the flag costs a DRAM round trip of its own)
    // the row is read piecemeal through references below: pull what will be read towards the SM now --
    // the observation runs if the observation is made of runs (the whole 10 KB row used to be fetched:
    // 348 MB per launch of 32 768 environments, two thirds of it never read), else the whole row
    if (g.n_obs_runs > 0) {
        for (int r = 0; r < g.n_obs_runs; ++r) {
            const char* p0 = reinterpret_cast<const char*>(S + g.obs_runs[3 * r]);
            const int bytes = g.obs_runs[3 * r + 2] * 8;
            for (int off = cx.tid * 128; off < bytes + 127; off += T * 128)
                asm volatile("prefetch.global.L2 [%0];" ::"l"(p0 + (off < bytes ? off : bytes - 1)));
        }
    } else {
        for (int off = cx.tid * 128; off < g.n_state * 8; off += T * 128)
            asm volatile("prefetch.global.L2 [%0];" ::"l"(reinterpret_cast<const char*>(S) + off));
    }
#endif
    const bool conv = B.converged[env] != 0;
    const double base = g.base_mva;
    const double* yv = yval_env ? yval_env : g.y_val;

    if (!conv) {
        // opf_env.py:390-399: NaN observation and reward, every constraint reported violated
        for (int j = cx.tid; j < g.n_obs; j += T) {
            if (B.obs_f32) B.obs_f32[env * (int64_t)g.n_obs + j] = NAN;
            if (B.obs_f64) B.obs_f64[env * (int64_t)g.n_obs + j] = NAN;
        }
        for (int c = cx.tid; c < nc; c += T) {
            if (B.valids) B.valids[env * nc + c] = 0;
            if (B.violations) B.violations[env * nc + c] = 1.0;
            if (B.penalties) B.penalties[env * nc + c] = 1.0;
        }
        if (cx.tid == 0) {
            if (B.reward) B.reward[env] = NAN;
            if (B.objective) B.objective[env] = NAN;
            if (B.penalty) B.penalty[env] = (double)nc;
            if (B.cost) B.cost[env] = NAN;
#ifdef OPFG_DEVICE_BUILD
            if (stats) atomicAdd(stats + OPFG_STAT_N, 1.0);
#else
            if (stats) stats[OPFG_STAT_N] += 1.0;
#endif
        }
        return;
    }

    // four buses per lane and trip: all eight loads are requested before the first sincos waits for one
    // (one DRAM round trip per trip instead of four; 17 % of this kernel's stall samples sat on these loads)
    for (int i0 = cx.tid; i0 < nb; i0 += 4 * T) {
        double m4[4], a4[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * T;
            m4[u] = i < nb ? vm[i] : 1.0;
            a4[u] = i < nb ? va[i] : 0.0;
        }
#pragma unroll
        for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * T;
            if (i >= nb) break;
            double sn, cs;
            const bool dead = g.isl && m4[u] != m4[u];      // dropped bus (island): V = 0 towards its neighbours, NaN results
            sincos(dead ? 0.0 : a4[u], &sn, &cs);
            s.vm[i] = m4[u];
            s.vr[i] = dead ? 0.0 : m4[u] * cs;
            s.vi[i] = dead ? 0.0 : m4[u] * sn;
        }
    }
    cx.sync();
    // branch flows and loading (pfsoln + results_branch.py [ext-mem], SURVEY.md App. B.5)
    const double* bry_env = (g.n_dyn > 0 && B.bry) ? B.bry + env * (int64_t)g.n_dyn * 8 : nullptr;
    for (int l = cx.tid; l < nbr; l += T) {
        const double* y = g.br_y + 8 * (size_t)l;
        bool half_open = false;
        if (bry_env) {
            const int d = g.dyn_of_branch[l];
            if (d >= 0) {                 // out of service (cell or switches): kernel 1 left no admittance at all
                y = bry_env + 8 * (size_t)d;
                const bool in_service = !(y[0] == 0.0 && y[1] == 0.0 && y[6] == 0.0 && y[7] == 0.0);
                half_open = in_service && y[2] == 0.0 && y[3] == 0.0;     // hangs from one end (open switch at the other)
            }
        }
        const int f = g.br_f[l], t = g.br_t[l];
        const double vfr = s.vr[f], vfi = s.vi[f], vtr = s.vr[t], vti = s.vi[t];
        const double ifr = y[0] * vfr - y[1] * vfi + y[2] * vtr - y[3] * vti;
        const double ifi = y[0] * vfi + y[1] * vfr + y[2] * vti + y[3] * vtr;
        const double itr = y[4] * vfr - y[5] * vfi + y[6] * vtr - y[7] * vti;
        const double iti = y[4] * vfi + y[5] * vfr + y[6] * vti + y[7] * vtr;
        const double pf = (vfr * ifr + vfi * ifi) * base, qf = (vfi * ifr - vfr * ifi) * base;
        const double pt = (vtr * itr + vti * iti) * base, qt = (vti * itr - vtr * iti) * base;
        const double lf = sqrt(pf * pf + qf * qf) * g.rate_f[l] / s.vm[f];
        const double lt = sqrt(pt * pt + qt * qt) * g.rate_t[l] / s.vm[t];
        const int slot = g.br_loading_slot[l];
        // pandapower: max(i_from, i_to) / i_max with numpy's NaN-propagating max (an end on a dropped bus: NaN); a
        // branch that is out of service has zero flows (its ppc rows are never written) -> 0 between live buses
        double ld = (lf != lf || lt != lt) ? NAN : (lf > lt ? lf : lt);
        if (half_open) ld = (y[0] != 0.0 || y[1] != 0.0) ? lf : lt;      // the open end sits on pandapower's auxiliary bus: no current
        if (slot >= 0) S[slot] = 100.0 * ld;
        const int fs = g.br_flow_slot[l];
        if (fs >= 0) { S[fs] = pf; S[fs + 1] = qf; S[fs + 2] = pt; S[fs + 3] = qt; }
    }
    // bus results in pandapower bus order (fused buses repeat their value)
    if (g.res_vm_slot >= 0)
        for (int b = cx.tid; b < g.n_pp_bus; b += T) {
            const int i = g.pp_lookup[b];
            S[g.res_vm_slot + b] = i >= 0 ? s.vm[i] : NAN;    // the copy in shared memory: no second trip to L2
            if (g.res_va_slot >= 0) S[g.res_va_slot + b] = i >= 0 ? va[i] * (180.0 / M_PI) : NAN;
        }
    // generator results: slack P, and Q of every voltage-controlled generator
    for (int gi = cx.tid; gi < g.ng; gi += T) {
        const int ps = g.gen_p_slot[gi], qs = g.gen_q_slot[gi];
        if (ps < 0 && qs < 0) continue;
        const int bus = g.gen_bus[gi];
        const int i = g.int_of_bus[bus];
        double ir = 0, ii = 0;
        for (int e = g.y_ptr[i]; e < g.y_ptr[i + 1]; ++e) {
            const int j = g.bus_of_int[g.y_meta[e].x & 0xffffu];
            ir += yv[2 * e] * s.vr[j] - yv[2 * e + 1] * s.vi[j];
            ii += yv[2 * e] * s.vi[j] + yv[2 * e + 1] * s.vr[j];
        }
        double P = s.vr[bus] * ir + s.vi[bus] * ii, Q = s.vi[bus] * ir - s.vr[bus] * ii;
        if (g.isl && s.vm[bus] != s.vm[bus]) P = Q = NAN;     // generator on a dropped bus
        if (ps >= 0) S[ps] = (P - sbus[2 * bus]) * base;
        if (qs >= 0) S[qs] = (Q - sbus[2 * bus + 1]) * base * g.gen_q_share[gi];
    }
    cx.sync();
#ifdef OPFG_DEVICE_BUILD
    __threadfence_block();
#endif
    if (g.n_t3 > 0) {
        // three-winding transformers (results_branch.py _get_trafo3w_results [ext-mem]): the branch loop above
        // left the loading at the outer end of each of the three star branches in three consecutive cells (the
        // star ends have factor 0); one element per lane takes the largest, NaN if any is NaN (numpy's max)
        for (int k = cx.tid; k < g.n_t3; k += T) {
            const double* c = S + g.t3_row_slot[k];
            const double a = c[0], b = c[1], d = c[2];
            S[g.t3_loading_slot[k]] = (a != a || b != b || d != d) ? NAN : fmax(a, fmax(b, d));
        }
        cx.sync();
#ifdef OPFG_DEVICE_BUILD
        __threadfence_block();
#endif
    }
    // constraints (opfgym/constraints.py:70-128)
    double pen_sum = 0;
    bool all_valid = true;
    for (int c = 0; c < nc; ++c) {
        // only_worst_case_violations (constraints.py:77-80, 113-122): the worst upper-bound violation
        // PLUS the worst lower-bound violation -- two running maxima, added after the reduction
        double viol = 0, viol_lo = 0, cnt = 0;
        const bool worst = g.con_worst[c] != 0;
        auto test = [&](double v, double hi, double lo) {
            if (v > hi) { const double x = fabs(v - hi); viol = worst ? (x > viol ? x : viol) : viol + x; cnt += 1; }
            if (v < lo) { const double x = fabs(v - lo); if (worst) viol_lo = x > viol_lo ? x : viol_lo; else viol += x; cnt += 1; }
        };
        int e = g.con_ptr[c] + cx.tid;
        const int e_end = g.con_ptr[c + 1];
        for (; e + T < e_end; e += 2 * T) {          // two entries per trip: their loads overlap
            const int f = e + T;
            const double v0 = ref_val(g, S, g.con_value[e]) * g.con_value_scale[e], m0 = g.con_bound_mul[e];
            const double v1 = ref_val(g, S, g.con_value[f]) * g.con_value_scale[f], m1 = g.con_bound_mul[f];
            const double hi0 = ref_val(g, S, g.con_max[e]) * m0, lo0 = ref_val(g, S, g.con_min[e]) * m0;
            const double hi1 = ref_val(g, S, g.con_max[f]) * m1, lo1 = ref_val(g, S, g.con_min[f]) * m1;
            test(v0, hi0, lo0);
            test(v1, hi1, lo1);
        }
        for (; e < e_end; e += T) {
            const double mul = g.con_bound_mul[e];
            test(ref_val(g, S, g.con_value[e]) * g.con_value_scale[e], ref_val(g, S, g.con_max[e]) * mul,
                 ref_val(g, S, g.con_min[e]) * mul);
        }
        cnt = cx.block_sum(cnt);
        viol = worst ? cx.block_max(viol) + cx.block_max(viol_lo) : cx.block_sum(viol);
        viol *= g.con_autoscale[c];
        const double pp = g.con_ppower[c];
        const double vp = pp == 1.0 ? viol : (pp == 2.0 ? viol * viol : pow(viol, pp));   // pow() is ~100 instructions
        const double pen = -(vp * g.con_pfactor[c] + cnt * g.con_pcount[c]);
        pen_sum += pen;
        if (cnt > 0) all_valid = false;
        if (cx.tid == 0) {
            if (B.valids) B.valids[env * nc + c] = cnt > 0 ? 0 : 1;
            if (B.violations) B.violations[env * nc + c] = viol;
            if (B.penalties) B.penalties[env * nc + c] = pen;
#ifdef OPFG_DEVICE_BUILD
            if (stats && cnt > 0 && c < OPFG_N_STATS - OPFG_STAT_VIOLATED0) atomicAdd(stats + OPFG_STAT_VIOLATED0 + c, 1.0);
#else
            if (stats && cnt > 0 && c < OPFG_N_STATS - OPFG_STAT_VIOLATED0) stats[OPFG_STAT_VIOLATED0 + c] += 1.0;
#endif
        }
    }
    // objective = -sum(costs)  (opfgym/objective.py:6-87, opf_env.py:493-500,517)
    double csum = 0;
    for (int r = cx.tid; r < g.n_poly; r += T) {
        const double p = ref_val(g, S, g.poly_p[r]) * g.poly_p_mul[r];
        const double q = ref_val(g, S, g.poly_q[r]) * g.poly_q_mul[r];
        const int* cf = g.poly_coef + 6 * (size_t)r;
        csum += ref_val(g, S, cf[0]) + ref_val(g, S, cf[1]) * p + ref_val(g, S, cf[2]) * p * p;
        csum += ref_val(g, S, cf[3]) + ref_val(g, S, cf[4]) * q + ref_val(g, S, cf[5]) * q * q;
    }
    for (int r = cx.tid; r < g.n_pwl; r += T)
        csum += pwl_cost(g, S, r, ref_val(g, S, g.pwl_v[r]) * g.pwl_v_mul[r]);
    const double objective = -cx.block_sum(csum) - (B.objective_offset ? B.objective_offset[env] : 0.0);
    // reward (opfgym/reward.py:61-98 and subclasses, SURVEY.md App. A.5)
    if (cx.tid == 0) {
        double obj = objective, pen = pen_sum;
        if (g.reward_kind == OPFG_REWARD_REPLACEMENT) obj = all_valid ? obj + g.valid_reward : 0.0;
        else if (g.reward_kind == OPFG_REWARD_PARAMETERIZED) {
            pen = all_valid ? pen + g.valid_reward : pen - g.invalid_penalty;
            if (!all_valid) obj *= g.invalid_obj_share;
        } else if (g.reward_kind == OPFG_REWARD_ONLY_OBJECTIVE) pen = 0.0;
        obj = obj * g.obj_factor + g.obj_bias;
        pen = pen * g.pen_factor + g.pen_bias;
        const double w = g.penalty_weight;
        double r = (w != w) ? obj + pen : obj * (1.0 - w) + pen * w;
        if (g.clip_lo == g.clip_lo) r = r < g.clip_lo ? g.clip_lo : (r > g.clip_hi ? g.clip_hi : r);
        double cost = all_valid ? 0.0 : fabs(pen_sum * g.pen_factor);
        if (!all_valid && g.reward_kind == OPFG_REWARD_PARAMETERIZED) cost += g.invalid_penalty;
        if (B.reward) B.reward[env] = r;
        if (B.objective) B.objective[env] = objective;
        if (B.penalty) B.penalty[env] = pen_sum;
        if (B.cost) B.cost[env] = cost;
        if (stats) {
            const double it = B.iterations ? (double)B.iterations[env] : 0.0;
#ifdef OPFG_DEVICE_BUILD
            atomicAdd(stats + OPFG_STAT_N, 1.0);
            atomicAdd(stats + OPFG_STAT_CONVERGED, 1.0);
            if (all_valid) atomicAdd(stats + OPFG_STAT_VALID, 1.0);
            atomicAdd(stats + OPFG_STAT_SUM_REWARD, r);
            atomicAdd(stats + OPFG_STAT_SUM_REWARD_SQ, r * r);
            atomicAdd(stats + OPFG_STAT_SUM_OBJECTIVE, objective);
            atomicAdd(stats + OPFG_STAT_SUM_PENALTY, pen_sum);
            atomicAdd(stats + OPFG_STAT_SUM_ITERS, it);
#else
            stats[OPFG_STAT_N] += 1.0; stats[OPFG_STAT_CONVERGED] += 1.0;
            if (all_valid) stats[OPFG_STAT_VALID] += 1.0;
            stats[OPFG_STAT_SUM_REWARD] += r; stats[OPFG_STAT_SUM_REWARD_SQ] += r * r;
            stats[OPFG_STAT_SUM_OBJECTIVE] += objective; stats[OPFG_STAT_SUM_PENALTY] += pen_sum;
            stats[OPFG_STAT_SUM_ITERS] += it;
#endif
        }
    }
    gather_obs(g, cx, S, B, env);
}

// ------------------------------------------------------------------------ Philox
OPFG_HD void philox4x32_10(uint32_t c0, uint32_t c1, uint32_t c2, uint32_t c3, uint32_t k0, uint32_t k1,
                           uint32_t* out) {
    for (int r = 0; r < 10; ++r) {
        const uint64_t p0 = (uint64_t)0xD2511F53u * c0, p1 = (uint64_t)0xCD9E8D57u * c2;
        const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c1 ^ k0, n1 = (uint32_t)p1;
        const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c3 ^ k1, n3 = (uint32_t)p0;
        c0 = n0; c1 = n1; c2 = n2; c3 = n3;
        k0 += 0x9E3779B9u; k1 += 0xBB67AE85u;
    }
    out[0] = c0; out[1] = c1; out[2] = c2; out[3] = c3;
}

// two doubles in [0,1) with 53 random bits each (numpy's uint64 -> double rule)
OPFG_HD void philox_two_doubles(uint64_t seed, uint64_t env, uint64_t stream, uint32_t pair, double* a, double* b) {
    uint32_t o[4];
    philox4x32_10(pair, (uint32_t)env, (uint32_t)(env >> 32), (uint32_t)stream ^ (uint32_t)(stream >> 32) * 0x9E3779B9u,
                  (uint32_t)seed, (uint32_t)(seed >> 32), o);
    const uint64_t x = ((uint64_t)o[1] << 32) | o[0], y = ((uint64_t)o[3] << 32) | o[2];
    *a = (double)(x >> 11) * (1.0 / 9007199254740992.0);
    *b = (double)(y >> 11) * (1.0 / 9007199254740992.0);
}

}  // namespace opfg
