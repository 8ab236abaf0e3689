// C ABI of libopfg_b200.so (see include/opfg_b200.h) and the CUDA kernels that
// wrap the per-environment algorithms of opfg_core.h: one CTA per environment,
// environment working set in shared memory, shared read-only grid tables read
// through L1/L2.
//
// Built twice:  nvcc -gencode arch=compute_100a,code=sm_100a  -> the product;
//               g++ -x c++ -DOPFG_HOSTSIM                       -> tests/hostsim only.
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <atomic>
#include <map>
#include <mutex>
#include <cmath>
#include <stdexcept>
#include <string>
#include <memory>
#include <vector>

#include "opfg_core.h"
#include "symbolic.hpp"

#ifndef OPFG_HOSTSIM
#include <cuda_runtime.h>
#endif

using namespace opfg;

namespace {

thread_local std::string g_error;
std::atomic<int64_t> g_launches{0};

int fail(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
    return -1;
}

// ------------------------------------------------------------- memory helpers
void* dev_alloc(size_t bytes) {
    if (bytes == 0) bytes = 8;
#ifdef OPFG_HOSTSIM
    return calloc(1, bytes);
#else
    void* p = nullptr;
    if (cudaMalloc(&p, bytes) != cudaSuccess) return nullptr;
    cudaMemset(p, 0, bytes);
    return p;
#endif
}
void dev_free(void* p) {
#ifdef OPFG_HOSTSIM
    free(p);
#else
    cudaFree(p);
#endif
}
void dev_put(void* dst, const void* src, size_t bytes) {
    if (!bytes) return;
#ifdef OPFG_HOSTSIM
    memcpy(dst, src, bytes);
#else
    cudaMemcpy(dst, src, bytes, cudaMemcpyHostToDevice);
#endif
}
void dev_get(void* dst, const void* src, size_t bytes) {
    if (!bytes) return;
#ifdef OPFG_HOSTSIM
    memcpy(dst, src, bytes);
#else
    cudaMemcpy(dst, src, bytes, cudaMemcpyDeviceToHost);
#endif
}

// Function attributes (dynamic shared-memory limit) are per DEVICE: remember what was raised per (device, kernel), so
// that a process driving several GPUs (envs on different devices, mixed-batch members) raises it on each of them
// (round-1 advisor finding: the bookkeeping used to live in process-wide statics).
#ifndef OPFG_HOSTSIM
template <class F>
void ensure_dynamic_smem(F* fn, size_t bytes) {
    if (bytes <= 48 * 1024) return;
    int dev = 0;
    cudaGetDevice(&dev);
    static std::mutex mu;
    static std::map<std::pair<int, const void*>, size_t> raised;
    std::lock_guard<std::mutex> lock(mu);
    size_t& cur = raised[{dev, reinterpret_cast<const void*>(fn)}];
    if (bytes > cur) {
        cudaFuncSetAttribute(fn, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        cur = bytes;
    }
}
int current_sm_count() {
    int dev = 0, n = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    return n;
}
#endif

}  // namespace

struct OpfgGrid {
    GridDev d{};
    Symbolic sym;
    OpfgGridDesc desc{};
    std::vector<void*> allocs;
    std::vector<int> gen_bus_host;
    std::vector<double> gen_q_share_host;
    std::vector<double> vm_bus_host;       // start |V| by ppc bus (set-point at generator buses)
    std::vector<int> br_f_host, br_t_host, type_host;     // ppc branch ends / bus types (island analysis)
    std::vector<unsigned char> br_on_host;                // static branch status
    std::vector<double> br_tap_host;                      // static off-nominal ratio
    int n_crit = 0;                                       // dynamic branches on the spanning tree (island analysis)
    int n_result_cells = 0;
    double flops_score = 0;
    bool has_assembly = false, has_scoring = false;
    int act_ref_max = -1, obs_ref_max = -1;   // largest state cell the action / observation tables touch
    size_t smem_pf = 0, smem_score = 0;
    int n_blocks_sym = 0;          // blocks of the filled Jacobian (d.n_blocks counts storage slots)
    int envs_per_cta = 1;
    int stage_level = 0;           // k_pf_multi: 0 = hot tables staged, 1 = + warm, 2 = all (OPFG_HOT/WARM/COLD_TABLES)
    // lane-per-environment kernel: schedule, per-warp scratch in global memory, launch shape
    LaneSchedule lane;
    int pf_kernel = 0;              // OpfgGridDesc.pf_kernel
    bool lanes_ok = false;          // tables built (the grid qualifies)
    double* lane_scratch = nullptr;
    size_t lane_warp_doubles = 0;   // scratch doubles per warp (32 lanes)
    int lane_ctas = 0, lane_warps_per_cta = 0, lane_stage = 0;
    size_t lane_smem = 0;
    bool lane_attr_set = false;
    int n_sm = 148;
    // fused kernel for radial grids: lanes per environment, environments per CTA, shared memory
    int tree_T = 0, tree_E = 0;
    size_t tree_env_doubles = 0, tree_smem = 0;
    bool tree_attr_set = false;

    // schedule / Ybus tables of the power-flow kernel live in ONE contiguous device arena so that a
    // multi-environment CTA can stage them in shared memory with a single cooperative copy
    char* tab_base = nullptr;
    size_t tab_cap = 0, tab_used = 0;
    void tab_reserve(size_t bytes) {
        tab_base = (char*)dev_alloc(bytes);
        if (!tab_base) throw std::runtime_error("device allocation failed");
        allocs.push_back(tab_base);
        tab_cap = bytes;
    }
    template <class T>
    T* tab(const std::vector<T>& v) {
        tab_used = (tab_used + 15) & ~size_t(15);
        const size_t bytes = v.size() * sizeof(T);
        if (tab_used + bytes > tab_cap) throw std::runtime_error("table arena overflow");
        char* p = tab_base + tab_used;
        dev_put(p, v.data(), bytes);
        tab_used += bytes;
        return (T*)p;
    }

    char* tab2_base = nullptr;
    size_t tab2_cap = 0, tab2_used = 0;
    template <class T>
    const T* tab2(const T* src, size_t n, bool from_device = false) {
        tab2_used = (tab2_used + 15) & ~size_t(15);
        const size_t bytes = n * sizeof(T);
        if (tab2_used + bytes > tab2_cap) throw std::runtime_error("scoring table arena overflow");
        char* p = tab2_base + tab2_used;
        if (bytes) {
#ifdef OPFG_HOSTSIM
            memcpy(p, src, bytes);
#else
            cudaMemcpy(p, src, bytes, from_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice);
#endif
        }
        tab2_used += bytes;
        return (const T*)p;
    }
    template <class T>
    const T* tab2(const std::vector<T>& v) { return tab2(v.data(), v.size()); }
    std::vector<double> consts_host;
    int score_threads = 32;

    template <class T>
    const T* up(const std::vector<T>& v) {
        void* p = dev_alloc(v.size() * sizeof(T));
        if (!p) throw std::runtime_error("device allocation failed");
        allocs.push_back(p);
        dev_put(p, v.data(), v.size() * sizeof(T));
        return (const T*)p;
    }
    template <class T>
    const T* up(const T* src, size_t n) {
        return up(std::vector<T>(src, src + n));
    }
    ~OpfgGrid() {
        for (void* p : allocs) dev_free(p);
    }
};

struct OpfgRowProgram {
    int n_rows = 0, n_ops = 0, n_regs = 1;
    int n_items = 0;                 // rows the program runs on (all of them, or the selected subset)
    int max_a = -1;                  // largest column start of a LOAD_STATE / STORE_STATE (-1: none)
    int max_cell = -1;               // largest state cell the program touches on its items
    int32_t* rows = nullptr;         // device, [n_items] table row of every item; null = item i is row i
    std::vector<int> host_rows;
    OpfgRowOp* ops = nullptr;        // device
    double* statics = nullptr;       // device
    std::vector<OpfgRowOp> host_ops;
    std::vector<double> host_statics;
    ~OpfgRowProgram() { dev_free(ops); dev_free(statics); dev_free(rows); }
};

// `r` is the program's register file, register i at r[i * rs]: a shared-memory column per thread in
// the CUDA build (a per-thread local array would be 128 B x 2 048 threads per SM -- it spills out of
// L1 and the interpreter ends up bound by local-memory traffic), a plain array in the host build.
OPFG_HHD void row_program_exec(const OpfgRowOp* ops, int n_ops, const double* statics, int row, double* S, double* r,
                               int rs) {
    for (int i = 0; i < n_ops; ++i) {
        const OpfgRowOp o = ops[i];
        switch (o.op) {
            case OPFG_OP_LOAD_STATE: r[o.dst * rs] = S[o.a + row]; break;
            case OPFG_OP_LOAD_STATIC: r[o.dst * rs] = statics[o.a + row]; break;
            case OPFG_OP_CONST: r[o.dst * rs] = o.imm; break;
            case OPFG_OP_ADD: r[o.dst * rs] = r[o.a * rs] + r[o.b * rs]; break;
            case OPFG_OP_SUB: r[o.dst * rs] = r[o.a * rs] - r[o.b * rs]; break;
            case OPFG_OP_MUL: r[o.dst * rs] = r[o.a * rs] * r[o.b * rs]; break;
            case OPFG_OP_DIV: r[o.dst * rs] = r[o.a * rs] / r[o.b * rs]; break;
            case OPFG_OP_SQRT: r[o.dst * rs] = sqrt(r[o.a * rs]); break;
            case OPFG_OP_NEG: r[o.dst * rs] = -r[o.a * rs]; break;
            case OPFG_OP_MIN: r[o.dst * rs] = fmin(r[o.a * rs], r[o.b * rs]); break;
            case OPFG_OP_MAX: r[o.dst * rs] = fmax(r[o.a * rs], r[o.b * rs]); break;
            case OPFG_OP_ABS: r[o.dst * rs] = fabs(r[o.a * rs]); break;
            case OPFG_OP_STORE_STATE: S[o.a + row] = r[o.b * rs]; break;
            default: break;
        }
    }
}

// OpfEnv._set_simbench_state for one cell (opf_env.py:317-372): profile row of the environment's time
// step, optional interpolation towards the next step, multiplicative uniform or additive normal
// noise, clipped to the profile's range.  Random numbers: element j of the Philox row of this
// environment (uniform noise: row of n_cols; normal noise: row of 2 n_cols, Box-Muller of j and n_cols + j).
OPFG_HD double profile_value(uint64_t seed, uint64_t env, uint64_t stream, int j, int n_cols, const double* table,
                              int n_steps, int64_t step, const double* r, const double* pmin, const double* pmax,
                              double noise_factor, int noise_kind) {
    double v = table[step * (int64_t)n_cols + j];
    if (r) {
        const int64_t nxt = step + 1 < n_steps ? step + 1 : n_steps - 1;
        v = v * r[0] + table[nxt * (int64_t)n_cols + j] * (1.0 - r[0]);
    }
    if (noise_kind == 1) {
        double u[2];
        philox_two_doubles(seed, env, stream, (uint32_t)(j >> 1), &u[0], &u[1]);
        v = v * (u[j & 1] * (2.0 * noise_factor) + (1.0 - noise_factor));
    } else if (noise_kind == 2) {
        double a[2], c[2];
        philox_two_doubles(seed, env, stream, (uint32_t)(j >> 1), &a[0], &a[1]);
        philox_two_doubles(seed, env, stream, (uint32_t)((n_cols + j) >> 1), &c[0], &c[1]);
        const double z = sqrt(-2.0 * log1p(-a[j & 1])) * cos(2.0 * M_PI * c[(n_cols + j) & 1]);
        v = v + fabs(v) * noise_factor * z;
    }
    return fmin(fmax(v, pmin[j]), pmax[j]);
}

// one stage of a fused episode reset (device form of OpfgResetStage)
struct ResetStage {
    int kind, n_cols;
    const int* slots;
    const double *lo, *hi, *dv;
    unsigned stream_off;
    const OpfgRowOp* ops;
    int n_ops, n_rows;
    const int32_t* rows;   // table row of every item (null: identity)
    const double* statics;
    int sync_after;      // 0: the next stage touches other cells and runs beside this one
    int item_off;        // first thread of this stage within its group (spreads the group's items)
    int ops_smem;        // offset (in OpfgRowOp units) of the staged copy of `ops`
};
struct OpfgResetPlan {
    std::vector<ResetStage> host;
    std::vector<std::vector<int>> reads, writes;     // per stage: state cells read / written
    ResetStage* dev = nullptr;
    int max_cell = -1, n_ops_total = 0, n_regs = 1;
    // decided per state layout (n_inputs) at the first launch
    int for_inputs = -1;
    bool covers_all = false;
    ~OpfgResetPlan() { dev_free(dev); }
};

// OpfEnv.reset for one environment (opf_env.py:180-220): sampler stages + hook programs, initial
// action, set-points, observation.  `S` is the environment's state row -- in the CUDA build a
// shared-memory copy of its input part, so every stage reads what the previous one wrote at
// shared-memory latency and the row goes to HBM once, coalesced.
template <class C>
OPFG_HD void env_reset(const GridDev& g, const C& cx, const OpfgBatch& B, int64_t env, double* S, const ResetStage* st,
                       int n_st, const OpfgRowOp* ops_staged, double* regs, int reg_stride, uint64_t seed, uint64_t first_env, uint64_t stream_base,
                       int random_action, unsigned action_stream_off) {
    const int T = cx.nthreads();
    for (int k = 0; k < n_st; ++k) {
        const ResetStage& s = st[k];
        const int first = (cx.tid + T - s.item_off % T) % T;
        if (s.kind == 0) {
            for (int pr = first; pr < (s.n_cols + 1) / 2; pr += T) {
                double u[2];
                philox_two_doubles(seed, first_env + (uint64_t)env, stream_base + s.stream_off, (uint32_t)pr, &u[0], &u[1]);
                for (int h = 0; h < 2; ++h) {
                    const int j = 2 * pr + h;
                    if (j < s.n_cols) S[s.slots[j]] = (s.lo[j] + (s.hi[j] - s.lo[j]) * u[h]) / s.dv[j];
                }
            }
        } else {
            const OpfgRowOp* ops = ops_staged ? ops_staged + s.ops_smem : s.ops;
            for (int r = first; r < s.n_rows; r += T)
                row_program_exec(ops, s.n_ops, s.statics, s.rows ? s.rows[r] : r, S, regs, reg_stride);
        }
        if (s.sync_after) cx.sync();
    }
    // initial action (:201-207) and its set-points: thread j owns action j
    double* act = const_cast<double*>(B.actions) + env * (int64_t)g.n_act;   // receives the initial action
    for (int j = cx.tid; j < g.n_act; j += T) {
        double u[2] = {0.5, 0.5};
        if (random_action)
            philox_two_doubles(seed, first_env + (uint64_t)env, stream_base + action_stream_off, (uint32_t)(j >> 1), &u[0], &u[1]);
        act[j] = u[j & 1];
    }
    cx.sync();
    env_assemble(g, cx, act, S, (double*)nullptr, (double*)nullptr, (double*)nullptr, true);
    cx.sync();
    gather_obs(g, cx, S, B, env);
}

// one member of a mixed batch (several grids scored by one launch, see k_score_mixed)
struct MixedMember {
    GridDev g;
    OpfgBatch B;
    int cta_begin, cta_end;     // CTAs of this member
    int score_threads;          // 32: one warp per environment (4 per CTA); 128: the whole CTA
    int score_env_doubles;
};
constexpr int OPFG_MAX_MEMBERS = 8;

// ------------------------------------------------------------------- kernels
#ifndef OPFG_HOSTSIM
// Elementwise kernels.  A 256-thread block is split into 256/W environment lanes of W item lanes
// (W a power of two): blockIdx.x walks item chunks, blockIdx.y environment groups, and a thread keeps
// its item while it loops over environments -- no 64-bit division per thread (it used to cost more
// than the work itself), per-item table values loaded once.
struct ItemGrid { dim3 grid; int w_log2; };
static ItemGrid item_grid(int64_t n_env, int n_items) {
    int w_log2 = 0;
    while ((1 << w_log2) < n_items && w_log2 < 8) ++w_log2;
    const int W = 1 << w_log2, epb = 256 / W;
    const int64_t groups = (n_env + epb - 1) / epb;
    return {dim3((unsigned)((n_items + W - 1) / W), (unsigned)std::max<int64_t>(1, std::min<int64_t>(groups, 8192))), w_log2};
}
#define OPFG_ITEM_LOOP(item, env, n_env_, w_log2)                                                   \
    const int item = (int)(blockIdx.x << (w_log2)) + (int)(threadIdx.x & ((1u << (w_log2)) - 1u));  \
    const int64_t env_step_ = (int64_t)gridDim.y * (256 >> (w_log2));                               \
    for (int64_t env = (int64_t)blockIdx.y * (256 >> (w_log2)) + (threadIdx.x >> (w_log2)); env < (n_env_); env += env_step_)
__global__ void k_row_program(const OpfgRowOp* ops, int n_ops, const double* statics, int n_rows, const int32_t* rows,
                              int64_t n_env, double* state, int n_state, int w_log2) {
    extern __shared__ __align__(16) double regs[];      // [n_regs][256] register file, one column per thread
    __shared__ OpfgRowOp sops[96];
    for (int i = threadIdx.x; i < n_ops; i += blockDim.x) sops[i] = ops[i];
    __syncthreads();
    OPFG_ITEM_LOOP(row, env, n_env, w_log2)
        if (row < n_rows)
            row_program_exec(sops, n_ops, statics, rows ? rows[row] : row, state + env * (int64_t)n_state, regs + threadIdx.x, 256);
}
// One CTA per environment.  Dynamic shared memory: [n_row doubles: input part of the state row]
// [n_st stages][all row-program ops][n_regs x T register file]; n_row == 0 keeps the row in global
// memory (tables that reach beyond the input part).
template <int T>
__global__ void __launch_bounds__(T) k_reset(GridDev g, OpfgBatch B, const ResetStage* st, int n_st, int n_row,
                                             int copy_in, int n_ops_total, uint64_t seed, uint64_t first_env,
                                             uint64_t stream_base, int random_action, unsigned action_stream_off) {
    extern __shared__ __align__(16) double sm[];
    Ctx<T> cx{(int)threadIdx.x, nullptr, 0};
    const int64_t env = blockIdx.x;
    double* Sg = B.state + env * (int64_t)g.n_state;
    ResetStage* st_s = reinterpret_cast<ResetStage*>(sm + n_row);
    OpfgRowOp* ops_s = reinterpret_cast<OpfgRowOp*>(st_s + n_st);
    for (int i = threadIdx.x; i < n_st * (int)(sizeof(ResetStage) / 8); i += T)
        reinterpret_cast<double*>(st_s)[i] = reinterpret_cast<const double*>(st)[i];
    if (copy_in)
        for (int i = threadIdx.x; i < n_row; i += T) sm[i] = Sg[i];
    __syncthreads();
    for (int k = 0; k < n_st; ++k)
        if (st_s[k].kind == 1)
            for (int i = threadIdx.x; i < st_s[k].n_ops * 3; i += T)
                reinterpret_cast<double*>(ops_s + st_s[k].ops_smem)[i] = reinterpret_cast<const double*>(st_s[k].ops)[i];
    __syncthreads();
    double* regs = reinterpret_cast<double*>(ops_s + n_ops_total) + threadIdx.x;
    env_reset(g, cx, B, env, n_row ? sm : Sg, st_s, n_st, ops_s, regs, T, seed, first_env, stream_base, random_action, action_stream_off);
    if (n_row) {
        __syncthreads();
        for (int i = threadIdx.x; i < n_row; i += T) Sg[i] = sm[i];
    }
}
// DC start for all environments: va[b, bus_of_int[i]] = theta0[i] + sum_bus P[b, bus] * Binv_t[bus, i]
// with P[b, bus] = Re Sbus[b, bus] (rows of Binv_t for reference buses are zero).  128 environments x
// 64 angles per CTA, 8 x 4 per thread (32 FMAs per 8 shared-memory wavefronts: FP64-pipe bound, the
// 4 x 4 version was bound by the LSU pipe), K in slices of 16 buses through a three-stage cp.async
// pipeline.  Plain FP64 FMA: 1 Gflop is no work for tensor cores.
constexpr int DC_ENVS = 128, DC_ST = 3;
constexpr size_t DC_SMEM = DC_ST * (16 * (DC_ENVS + 2) + 16 * 64) * sizeof(double);
__global__ void __launch_bounds__(256, 2) k_dc_start(GridDev g, OpfgBatch B) {
    extern __shared__ __align__(16) double dc_sm[];
    double (*p_s)[16][DC_ENVS + 2] = reinterpret_cast<double (*)[16][DC_ENVS + 2]>(dc_sm);                   // [stage][bus][env]
    double (*b_s)[16][64] = reinterpret_cast<double (*)[16][64]>(dc_sm + DC_ST * 16 * (DC_ENVS + 2));     // [stage][bus][i]
    const int tx = threadIdx.x & 15, ty = threadIdx.x >> 4;          // angles tx + 16 c, environments 8 ty + a
    const int64_t env0 = (int64_t)blockIdx.x * DC_ENVS;
    const int i0 = blockIdx.y * 64, n = g.n, nb = g.nb;
    const int n_slices = (nb + 15) / 16;
    const int pe = threadIdx.x >> 4, pk = threadIdx.x & 15;         // P: environments pe + 16 r, bus pk
    const int bk = threadIdx.x >> 6, bi = threadIdx.x & 63;         // B: buses bk + 4 r, angle bi
    auto issue = [&](int slice) {
        if (slice < n_slices) {
            const int st = slice % DC_ST, k0 = slice * 16;
#pragma unroll
            for (int r = 0; r < DC_ENVS / 16; ++r) {
                const int e = pe + 16 * r;
                const int64_t env = env0 + e;
                double* dst = &p_s[st][pk][e];
                if (k0 + pk < nb && env < B.n_env) {
                    const double* src = B.sbus + (env * nb + k0 + pk) * 2;
                    asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(dst)), "l"(src));
                } else {
                    *dst = 0.0;
                }
            }
#pragma unroll
            for (int r = 0; r < 4; ++r) {
                const double* bsrc = g.dc_binv_t + (size_t)(k0 + bk + 4 * r) * g.dc_ld + i0 + bi;   // zero padded tiles
                asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"((unsigned)__cvta_generic_to_shared(&b_s[st][bk + 4 * r][bi])), "l"(bsrc));
            }
        }
        asm volatile("cp.async.commit_group;");
    };
    double acc[8][4] = {};
    issue(0);
    issue(1);
    for (int slice = 0; slice < n_slices; ++slice) {
        issue(slice + 2);
        asm volatile("cp.async.wait_group 2;");
        __syncthreads();
        const int st = slice % DC_ST;
#pragma unroll 4
        for (int kk = 0; kk < 16; ++kk) {
            double pv[8];
#pragma unroll
            for (int h = 0; h < 4; ++h) {
                const double2 t = *reinterpret_cast<const double2*>(&p_s[st][kk][ty * 8 + 2 * h]);
                pv[2 * h] = t.x; pv[2 * h + 1] = t.y;
            }
            // angles tx, tx+16, tx+32, tx+48: the 16 lanes of a row read 128 contiguous bytes per load
            const double bv[4] = {b_s[st][kk][tx], b_s[st][kk][tx + 16], b_s[st][kk][tx + 32], b_s[st][kk][tx + 48]};
#pragma unroll
            for (int a = 0; a < 8; ++a)
#pragma unroll
                for (int c = 0; c < 4; ++c) acc[a][c] = fma(pv[a], bv[c], acc[a][c]);
        }
        __syncthreads();                                    // the stage is refilled by the next issue()
    }
#pragma unroll
    for (int a = 0; a < 8; ++a) {
        const int64_t env = env0 + ty * 8 + a;
        if (env >= B.n_env) continue;
#pragma unroll
        for (int c = 0; c < 4; ++c) {
            const int i = i0 + tx + 16 * c;
            if (i < n) B.va[env * nb + g.bus_of_int[i]] = acc[a][c] + g.dc_theta0[i];
        }
    }
}
__global__ void k_branch_y(GridDev g) {
    const int l = blockIdx.x * blockDim.x + threadIdx.x;
    if (l < g.nbr) branch_admittance(g.br_param + 6 * (size_t)l, g.br_y + 8 * (size_t)l);
}
__global__ void k_ybus(GridDev g, double* y_val) {
    const int e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e < g.nnz_y) ybus_entry(g, g.br_y, e, y_val + 2 * (size_t)e);
}
__global__ void k_philox(uint64_t seed, uint64_t first_env, uint64_t stream, int64_t n_env, int n_cols, double* out,
                         int w_log2) {
    OPFG_ITEM_LOOP(pr, b, n_env, w_log2) {
        if (2 * pr >= n_cols) break;
        double u0, u1;
        philox_two_doubles(seed, first_env + (uint64_t)b, stream, (uint32_t)pr, &u0, &u1);
        double* row = out + b * (int64_t)n_cols;
        row[2 * pr] = u0;
        if (2 * pr + 1 < n_cols) row[2 * pr + 1] = u1;
    }
}
__global__ void k_sample_uniform(uint64_t seed, uint64_t first_env, uint64_t stream, int64_t n_env, int n_cols,
                                 const int* slots, const double* lo, const double* hi, const double* dv,
                                 double* state, int n_state, int w_log2, const int* obs_pos, float* o32, double* o64,
                                 int n_obs) {
    const int pr0 = (int)(blockIdx.x << w_log2) + (int)(threadIdx.x & ((1u << w_log2) - 1u));
    if (2 * pr0 >= n_cols) return;
    const int j0 = 2 * pr0, j1 = 2 * pr0 + 1;
    const bool two = j1 < n_cols;
    const int s0 = slots[j0], s1 = two ? slots[j1] : 0;
    const int p0 = obs_pos ? obs_pos[j0] : -1, p1 = (obs_pos && two) ? obs_pos[j1] : -1;
    const double lo0 = lo[j0], w0 = hi[j0] - lo0, d0 = dv[j0];
    const double lo1 = two ? lo[j1] : 0.0, w1 = two ? hi[j1] - lo1 : 0.0, d1 = two ? dv[j1] : 1.0;
    OPFG_ITEM_LOOP(pr, b, n_env, w_log2) {
        double u0, u1;
        philox_two_doubles(seed, first_env + (uint64_t)b, stream, (uint32_t)pr, &u0, &u1);
        double* row = state + b * (int64_t)n_state;
        const double v0 = (lo0 + w0 * u0) / d0, v1 = (lo1 + w1 * u1) / d1;
        row[s0] = v0;
        if (two) row[s1] = v1;
        if (p0 >= 0) { if (o32) o32[b * (int64_t)n_obs + p0] = (float)v0; else o64[b * (int64_t)n_obs + p0] = v0; }
        if (p1 >= 0) { if (o32) o32[b * (int64_t)n_obs + p1] = (float)v1; else o64[b * (int64_t)n_obs + p1] = v1; }
    }
}
__global__ void k_sample_profiles(uint64_t seed, uint64_t first_env, uint64_t stream, int64_t n_env, int n_cols,
                                  const int* slots, const double* table, int n_steps, const int64_t* step,
                                  const double* interp_r, const double* pmin, const double* pmax, double noise_factor,
                                  int noise_kind, double* state, int n_state, int w_log2) {
    OPFG_ITEM_LOOP(j, b, n_env, w_log2) {
        if (j >= n_cols) break;
        state[b * (int64_t)n_state + slots[j]] = profile_value(seed, first_env + (uint64_t)b, stream, j, n_cols, table, n_steps,
                                                               step[b], interp_r ? interp_r + b : nullptr, pmin, pmax,
                                                               noise_factor, noise_kind);
    }
}
// One warp per environment, two environments per CTA (lifts the 32-CTAs-per-SM limit on resident envs).
// Both kernels wait on DRAM loads behind references: more resident warps = more loads in flight.
// k_assemble_warps keeps the compiler's default for 128-thread bounds (62 registers); k_score_warps asks for 24
// two-warp CTAs per SM (40 registers).  Measured for k_score_warps (122-bus grid, 32 768 environments):
// 56 registers 234 us, 48 -> 217, 40 -> 210, 70 -> 254.
__global__ void __launch_bounds__(128) k_assemble_warps(GridDev g, OpfgBatch B) {
    const int64_t env = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (env >= B.n_env) return;
    Ctx<32> cx{(int)(threadIdx.x & 31), nullptr, 0};
    env_assemble(g, cx, B.actions ? B.actions + env * g.n_act : nullptr, B.state + env * (int64_t)g.n_state,
                 B.sbus ? B.sbus + env * (int64_t)g.nb * 2 : nullptr,
                 B.yval ? B.yval + env * (int64_t)g.nnz_y * 2 : nullptr,
                 B.bry ? B.bry + env * (int64_t)g.n_dyn * 8 : nullptr, B.absolute_actions != 0,
                 B.vm ? B.vm + env * (int64_t)g.nb : nullptr);
}
__global__ void __launch_bounds__(64, 24) k_score_warps(GridDev g, OpfgBatch B, int env_doubles) {
    extern __shared__ __align__(16) double sm[];
    const int64_t env = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (env >= B.n_env) return;
    double* mine = sm + (size_t)(threadIdx.x >> 5) * env_doubles;
    Ctx<32> cx{(int)(threadIdx.x & 31), mine + score_smem_doubles(g.nb, g.nbr, 32) - 4, 0};
    env_score(g, cx, mine, B, env, (g.n_dyn > 0 && B.yval) ? B.yval + env * (int64_t)g.nnz_y * 2 : nullptr,
              B.state + env * (int64_t)g.n_state);
}
// Mixed batch (BASELINE config 4): ONE launch of kernel 1 / kernel 5 over several grids.  Every CTA looks
// up its member (grid descriptor + batch, in device memory) from its block index; environments of
// different grids therefore run side by side in one grid of CTAs, each with its own tables.
__global__ void __launch_bounds__(128) k_assemble_mixed(const MixedMember* members, int n_members) {
    int m = 0;
    while (m + 1 < n_members && (int)blockIdx.x >= members[m].cta_end) ++m;
    const MixedMember& mm = members[m];
    const GridDev& g = mm.g;
    const OpfgBatch& B = mm.B;
    const int64_t env = (int64_t)(blockIdx.x - mm.cta_begin) * 4 + (threadIdx.x >> 5);
    if (env >= B.n_env) return;
    Ctx<32> cx{(int)(threadIdx.x & 31), nullptr, 0};
    env_assemble(g, cx, B.actions ? B.actions + env * g.n_act : nullptr, B.state + env * (int64_t)g.n_state,
                 B.sbus ? B.sbus + env * (int64_t)g.nb * 2 : nullptr,
                 B.yval ? B.yval + env * (int64_t)g.nnz_y * 2 : nullptr,
                 B.bry ? B.bry + env * (int64_t)g.n_dyn * 8 : nullptr, B.absolute_actions != 0,
                 B.vm ? B.vm + env * (int64_t)g.nb : nullptr);
}
__global__ void __launch_bounds__(128) k_score_mixed(const MixedMember* members, int n_members) {
    extern __shared__ __align__(16) double sm[];
    int m = 0;
    while (m + 1 < n_members && (int)blockIdx.x >= members[m].cta_end) ++m;
    const MixedMember& mm = members[m];
    const GridDev& g = mm.g;
    const OpfgBatch& B = mm.B;
    if (mm.score_threads == 32) {
        const int64_t env = (int64_t)(blockIdx.x - mm.cta_begin) * 4 + (threadIdx.x >> 5);
        if (env >= B.n_env) return;
        double* mine = sm + (size_t)(threadIdx.x >> 5) * mm.score_env_doubles;
        Ctx<32> cx{(int)(threadIdx.x & 31), mine + score_smem_doubles(g.nb, g.nbr, 32) - 4, 0};
        env_score(g, cx, mine, B, env, (g.n_dyn > 0 && B.yval) ? B.yval + env * (int64_t)g.nnz_y * 2 : nullptr,
                  B.state + env * (int64_t)g.n_state);
    } else {
        const int64_t env = blockIdx.x - mm.cta_begin;
        if (env >= B.n_env) return;
        Ctx<128> cx{(int)threadIdx.x, sm + score_smem_doubles(g.nb, g.nbr, 128) - 2 * (128 / 32 + 1), 0};
        env_score(g, cx, sm, B, env, (g.n_dyn > 0 && B.yval) ? B.yval + env * (int64_t)g.nnz_y * 2 : nullptr,
                  B.state + env * (int64_t)g.n_state);
    }
}

template <int T>
__global__ void __launch_bounds__(T) k_pf(GridDev g, OpfgBatch B) {
    extern __shared__ __align__(16) double sm[];
    const int64_t env = blockIdx.x;
    Ctx<T> cx{(int)threadIdx.x, sm + pf_smem_doubles(g.n_blocks, g.n, g.nb, T) - 2 * (T / 32 + 1) - 2, 0};
    env_pf_solve(g, cx, sm, B.sbus + env * (int64_t)g.nb * 2,
                 (g.n_dyn > 0 && B.yval) ? B.yval + env * (int64_t)g.nnz_y * 2 : nullptr, B.vm + env * (int64_t)g.nb,
                 B.va + env * (int64_t)g.nb, B.converged + env, B.iterations + env);
}
// Persistent multi-environment CTA: E environments of T threads each share ONE shared-memory copy of
// the schedule / Ybus tables (their reads are on the critical path of every level); each environment
// group synchronises on its own named barrier and walks through its share of the batch.
// Tables of the staged arena, in allocation order: the LU schedule and the Ybus index tables ("hot", always
// staged), the Ybus values ("warm", read in every iteration) and the start-value / q-limit tables ("cold",
// read once per solve).  STAGE = 0 stages the hot part, 1 hot + warm, 2 everything -- whichever lets
// the most environments share an SM.
#define OPFG_HOT_TABLES(X)                                                                      \
    X(bus_of_int) X(type_int) X(level_ptr) X(fill_ids) X(dp_ptr) X(dp_pack) X(dp_own) \
    X(eg_ptr) X(eg_item) X(off_ptr) X(off_hdr) X(op_pack) X(up_ptr) X(up_pack) X(y_ptr) X(y_meta)
#define OPFG_WARM_TABLES(X) X(y_val)
#define OPFG_COLD_TABLES(X) X(vm0_int) X(va0_int) X(qlim_bus) X(qlim_min) X(qlim_max)

// The kernel receives a view of GridDev in which every staged table pointer holds its BYTE OFFSET in
// the arena (staged_view below).  Adding the offset to the shared-memory base is one instruction and
// leaves the address space known to the compiler (LDS instead of generic loads); the earlier
// "if the pointer lies in the staged range, move it" form was re-evaluated at the use sites under
// the 96-register cap and cost 10 % of the kernel's instructions.
// MODE = STAGE | (4 if the Ybus values are per environment): with the shared table the compiler
// knows the values live in shared memory (LDS instead of generic loads in the row pass).
// BOUND: the largest block this instantiation is launched with (T x environments per CTA): 768 caps the kernel at
// 85 registers (it spills there), so launches of at most 384 / 256 threads get their own, roomier build
template <int T, int MODE, int BOUND = 768>
__global__ void __launch_bounds__(BOUND, 1) k_pf_multi(GridDev g, OpfgBatch B, int E, int env_doubles) {
    constexpr int STAGE = MODE & 3;
    constexpr bool DYN = (MODE & 4) != 0;
    extern __shared__ __align__(16) double sm[];
    {
        const int4* src = reinterpret_cast<const int4*>(g.tab_base);
        int4* dst = reinterpret_cast<int4*>(sm);
        for (int i = threadIdx.x; i < g.tab_staged_bytes / 16; i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    char* sbase = reinterpret_cast<char*>(sm);
#define OPFG_REBASE(field) g.field = reinterpret_cast<decltype(g.field)>(sbase + (unsigned)reinterpret_cast<size_t>(g.field));
    OPFG_HOT_TABLES(OPFG_REBASE)
    if (STAGE >= 1) { OPFG_WARM_TABLES(OPFG_REBASE) }
    if (STAGE >= 2) { OPFG_COLD_TABLES(OPFG_REBASE) }
#undef OPFG_REBASE
    const int e_local = threadIdx.x / T;
    double* mine = sm + g.tab_staged_bytes / 8 + (size_t)e_local * env_doubles;
    Ctx<T> cx{(int)(threadIdx.x % T), mine + pf_smem_doubles(g.n_blocks, g.n, g.nb, T) - 2 * (T / 32 + 1) - 2, 1 + e_local};
    // every CTA owns a contiguous share of the batch: the last, partial round is then spread over ALL SMs (a few
    // environments each, running faster for the lack of competition) instead of filling a quarter of them
    const int64_t lo = B.n_env * (int64_t)blockIdx.x / gridDim.x, hi = B.n_env * ((int64_t)blockIdx.x + 1) / gridDim.x;
    for (int64_t env = lo + e_local; env < hi; env += E) {
        env_pf_solve(g, cx, mine, B.sbus + env * (int64_t)g.nb * 2,
                     DYN ? B.yval + env * (int64_t)g.nnz_y * 2 : (const double*)nullptr,
                     B.vm + env * (int64_t)g.nb, B.va + env * (int64_t)g.nb, B.converged + env, B.iterations + env);
        cx.sync();
    }
}
// Fused kernel for radial grids (opfg_core.h, env_pf_tree): persistent CTAs, E environments of T lanes
// each (32 / T environments share a warp and run in lockstep), tables staged once per CTA.
#define OPFG_TREE_TABLES(X) X(tr_bus_of_int) X(tr_level_ptr) X(tr_y_ptr) X(tr_parent) X(tr_type) X(tr_y_ent) X(tr_y_val) X(tr_vm0) X(tr_va0)
template <int T, bool DYN, int MAX_THREADS>
__global__ void __launch_bounds__(MAX_THREADS, 1) k_pf_tree(GridDev g, OpfgBatch B, int E, int env_doubles) {
    extern __shared__ __align__(16) double sm[];
    {
        const int4* src = reinterpret_cast<const int4*>(g.tab4_base);
        int4* dst = reinterpret_cast<int4*>(sm);
        for (int i = threadIdx.x; i < g.tab4_bytes / 16; i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    char* sbase = reinterpret_cast<char*>(sm);
#define OPFG_REBASE(field) g.field = reinterpret_cast<decltype(g.field)>(sbase + (unsigned)reinterpret_cast<size_t>(g.field));
    OPFG_TREE_TABLES(OPFG_REBASE)
#undef OPFG_REBASE
    const int grp = threadIdx.x / T;
    double* mine = sm + g.tab4_bytes / 8 + (size_t)grp * env_doubles;
    Grp<T> cx{(int)(threadIdx.x % T)};
    // every CTA owns a contiguous share of the batch: the last, partial round is then spread over ALL SMs (a few
    // environments each, running faster for the lack of competition) instead of filling a quarter of them
    const int64_t lo = B.n_env * (int64_t)blockIdx.x / gridDim.x, hi = B.n_env * ((int64_t)blockIdx.x + 1) / gridDim.x;
    for (int64_t base = lo; base < hi; base += E) {
        if (base + (grp & ~(32 / T - 1)) >= hi) break;   // no environment left for this warp (the solve only uses __syncwarp)
        int64_t env = base + grp;
        const bool live = env < hi;
        if (!live) env = hi - 1;               // an idle group shadows its warp's last environment (no stores)
        env_pf_tree<Grp<T>, DYN>(g, cx, mine, B.sbus + env * (int64_t)g.nb * 2,
                    DYN ? B.yval + env * (int64_t)g.nnz_y * 2 : (const double*)nullptr,
                    B.vm + env * (int64_t)g.nb, B.va + env * (int64_t)g.nb, B.converged + env, B.iterations + env, live);
        __syncwarp();
    }
}
template <int T, int MODE>
static void (*pick_multi(int bound))(GridDev, OpfgBatch, int, int) {
    return bound == 256 ? k_pf_multi<T, MODE, 256> : (bound == 384 ? k_pf_multi<T, MODE, 384> : k_pf_multi<T, MODE, 768>);
}
static GridDev tree_view(const GridDev& d) {
    GridDev view = d;
#define OPFG_TO_OFFSET(field) view.field = reinterpret_cast<decltype(view.field)>((size_t)(reinterpret_cast<const char*>(d.field) - d.tab4_base));
    OPFG_TREE_TABLES(OPFG_TO_OFFSET)
#undef OPFG_TO_OFFSET
    return view;
}

// Lane-per-environment Newton-Raphson (opfg_core.h, lanes_pf_solve): persistent CTAs of W warps, a warp
// takes 32 consecutive environments at a time.  Shared memory: the schedule tables (staged once per
// CTA when STAGED, else read through L1) and one row buffer per warp; everything else per environment
// sits in the warp's scratch slice in global memory at [slot][lane].
#define OPFG_LANE_TABLES(X)                                                                   \
    X(ln_row) X(ln_y) X(ln_diag_pos) X(ln_fill) X(ln_el) X(ln_el_uptr) X(ln_upd) X(ln_up)     \
    X(ln_yval) X(ln_vm0) X(ln_va0) X(ln_bus_of_int) X(ln_type) X(ln_qbus) X(ln_qmin) X(ln_qmax)
// MODE bits: 1 = tables staged in shared memory, 2 = enforce_q_lims (per-lane bus types), 4 = per-environment Ybus values
template <int MODE>
__global__ void __launch_bounds__(512, 1) k_pf_lanes(GridDev g, OpfgBatch B, double* scratch, size_t warp_doubles) {
    constexpr bool STAGED = (MODE & 1) != 0, QLIM = (MODE & 2) != 0, DYN = (MODE & 4) != 0;
    extern __shared__ __align__(16) double sm[];
    size_t tab_doubles = 0;
    if (STAGED) {
        const int4* src = reinterpret_cast<const int4*>(g.tab3_base);
        int4* dst = reinterpret_cast<int4*>(sm);
        for (int i = threadIdx.x; i < g.tab3_bytes / 16; i += blockDim.x) dst[i] = src[i];
        __syncthreads();
        char* sbase = reinterpret_cast<char*>(sm);
#define OPFG_REBASE(field) g.field = reinterpret_cast<decltype(g.field)>(sbase + (unsigned)reinterpret_cast<size_t>(g.field));
        OPFG_LANE_TABLES(OPFG_REBASE)
#undef OPFG_REBASE
        tab_doubles = (size_t)g.tab3_bytes / 8;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpc = blockDim.x >> 5;
    double* rb = sm + tab_doubles + (size_t)warp * (4 * g.ln_max_row * 32) + lane;
    const size_t gwarp = (size_t)blockIdx.x * wpc + warp;
    const LaneMem<32> s = lane_carve<32>(scratch + gwarp * warp_doubles + lane, rb, g.nb, g.n, g.ln_n_up);
    const int64_t n_groups = (B.n_env + 31) / 32;
    for (int64_t grp = gwarp; grp < n_groups; grp += (int64_t)gridDim.x * wpc) {
        int64_t env = grp * 32 + lane;
        const bool live = env < B.n_env;
        if (!live) env = B.n_env - 1;          // idle lanes shadow the last environment (no stores)
        lanes_pf_solve<32, QLIM, DYN>(g, s, B.sbus + env * (int64_t)g.nb * 2,
                                      DYN ? B.yval + env * (int64_t)g.nnz_y * 2 : (const double*)nullptr,
                                      B.vm + env * (int64_t)g.nb, B.va + env * (int64_t)g.nb, B.converged + env,
                                      B.iterations + env, live);
        __syncwarp();
    }
}
static GridDev lane_view(const GridDev& d, bool staged) {
    GridDev view = d;
    if (staged) {
#define OPFG_TO_OFFSET(field) view.field = reinterpret_cast<decltype(view.field)>((size_t)(reinterpret_cast<const char*>(d.field) - d.tab3_base));
        OPFG_LANE_TABLES(OPFG_TO_OFFSET)
#undef OPFG_TO_OFFSET
    }
    return view;
}

template <int T>
__global__ void __launch_bounds__(T) k_score(GridDev g, OpfgBatch B) {
    extern __shared__ __align__(16) double sm[];
    const int64_t env = blockIdx.x;
    Ctx<T> cx{(int)threadIdx.x, sm + score_smem_doubles(g.nb, g.nbr, T) - 2 * (T / 32 + 1), 0};
    env_score(g, cx, sm, B, env, (g.n_dyn > 0 && B.yval) ? B.yval + env * (int64_t)g.nnz_y * 2 : nullptr,
              B.state + env * (int64_t)g.n_state);
}

__global__ void k_observe(GridDev g, OpfgBatch B, int w_log2) {
    OPFG_ITEM_LOOP(j, env, B.n_env, w_log2) {
        if (j >= g.n_obs) break;
        const double v = obs_value(g, B.state + env * (int64_t)g.n_state, j);
        if (B.obs_f32) B.obs_f32[env * (int64_t)g.n_obs + j] = (float)v;
        if (B.obs_f64) B.obs_f64[env * (int64_t)g.n_obs + j] = v;
    }
}

__global__ void __launch_bounds__(256) k_fp64_probe(int iters, double* out) {
    double a0 = threadIdx.x * 1e-9, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double m = 1.0000001, c = 1e-9;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, m, c); a1 = fma(a1, m, c); a2 = fma(a2, m, c); a3 = fma(a3, m, c);
        a4 = fma(a4, m, c); a5 = fma(a5, m, c); a6 = fma(a6, m, c); a7 = fma(a7, m, c);
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 12345.678) out[0] = s;   // never true; keeps the chains alive
}

// staged view of the grid for k_pf_multi: table pointers -> byte offsets in the arena
static GridDev staged_view(const GridDev& d, int stage) {
    GridDev view = d;
#define OPFG_TO_OFFSET(field) view.field = reinterpret_cast<decltype(view.field)>((size_t)(reinterpret_cast<const char*>(d.field) - d.tab_base));
    OPFG_HOT_TABLES(OPFG_TO_OFFSET)
    if (stage >= 1) { OPFG_WARM_TABLES(OPFG_TO_OFFSET) }
    if (stage >= 2) { OPFG_COLD_TABLES(OPFG_TO_OFFSET) }
#undef OPFG_TO_OFFSET
    return view;
}

#define OPFG_DISPATCH_T(T_, ...)                                     \
    switch (T_) {                                                    \
        case 32: { constexpr int TT = 32; __VA_ARGS__; break; }      \
        case 64: { constexpr int TT = 64; __VA_ARGS__; break; }      \
        case 128: { constexpr int TT = 128; __VA_ARGS__; break; }    \
        case 256: { constexpr int TT = 256; __VA_ARGS__; break; }    \
        default: return fail("unsupported threads_per_env %d", T_);  \
    }
#endif

// lanes per environment of the fused radial kernel (also the cap of its balanced levels).  Measured on
// the 122-bus grid with the centre-rooted order (B200 at 1000 W, 32 768 environments, opfg_pf_solve incl.
// the DC-start GEMM): 8 lanes 1.051 ms (17 levels), 16 lanes 0.758 ms (14 levels), 32 lanes 0.990 ms
// (14 levels, 16 environments per SM) -- the kernel is bound by the latency of its level chain, more lanes
// mean fewer rounds per level until the idle lanes of the narrow levels cost more issue slots than the
// rounds save.
constexpr int TREE_LANES = 16;

// Radial grid with the dense DC pre-pass: the fused kernel (pf_kernel 0 = auto or 3 = radial)
static bool use_tree(const OpfgGrid* G, const OpfgBatch* B) {
    (void)B;
    const GridDev& d = G->d;
    return d.tr_ok && (G->pf_kernel == 0 || G->pf_kernel == 3) && (!d.init_dc || d.dc_pre);
}

// Which power-flow kernel a launch uses: the lane-per-environment kernel when its tables exist (row
// patterns of at most 255 blocks, row buffer fits shared memory) and the DC start comes from the dense
// pre-pass; else one CTA per environment.  Only OpfgGridDesc.pf_kernel = 2 selects it.
static bool use_lanes(const OpfgGrid* G, const OpfgBatch* B) {
    (void)B;
    if (G->pf_kernel != 2) return false;
    const GridDev& d = G->d;
    return G->lanes_ok && G->lane_scratch && (!d.init_dc || d.dc_pre) && !d.isl;   // the lane kernel has no island handling
}

// ------------------------------------------------------------------- C ABI
extern "C" {

int opfg_version(void) { return OPFG_VERSION; }
const char* opfg_last_error(void) { return g_error.c_str(); }
int64_t opfg_launch_count(void) { return g_launches.load(); }

int opfg_grid_create(const OpfgGridDesc* desc, OpfgGrid** out) {
    if (!desc || !out) return fail("null argument");
    *out = nullptr;
    if (desc->nb <= 0 || !desc->bus || !desc->branch || !desc->gen) return fail("empty grid tables");
    if (desc->bus_cols < 10 || desc->gen_cols < 8 || desc->branch_cols < 11) return fail("ppc tables too narrow");
#ifndef OPFG_HOSTSIM
    {
        int ndev = 0;
        if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
            return fail("no CUDA device: libopfg_b200 has no CPU path");
    }
#endif
    try {
        auto* G = new OpfgGrid();
        G->desc = *desc;
        const int nb = desc->nb, nbr = desc->nbr, ng = desc->ng;
        const double base = desc->base_mva;
        std::vector<int> type(nb);
        std::vector<double> ysh(2 * (size_t)nb), va_ref(nb), vm_bus(nb);
        int n_ref = 0;
        for (int b = 0; b < nb; ++b) {
            const double* row = desc->bus + (size_t)b * desc->bus_cols;
            type[b] = (int)row[OPFG_BUS_TYPE];
            if (type[b] < 1 || type[b] > 3) { delete G; return fail("bus %d has unsupported type %d", b, type[b]); }
            n_ref += type[b] == 3;
            ysh[2 * b] = row[OPFG_GS] / base;
            ysh[2 * b + 1] = row[OPFG_BS] / base;
            vm_bus[b] = row[OPFG_VM];
            va_ref[b] = row[OPFG_VA] * M_PI / 180.0;
        }
        if (n_ref == 0) { delete G; return fail("grid has no reference bus"); }
        // generator set-points: V0[gbus] = VG (pandapower _get_pf_variables_from_ppci)
        std::vector<int> vgens(nb, 0);
        G->gen_bus_host.resize(ng);
        for (int gI = 0; gI < ng; ++gI) {
            const double* row = desc->gen + (size_t)gI * desc->gen_cols;
            const int bus = (int)row[OPFG_GEN_BUS];
            if (bus < 0 || bus >= nb) { delete G; return fail("generator %d on invalid bus", gI); }
            G->gen_bus_host[gI] = bus;
            if (row[OPFG_GEN_STATUS] > 0 && type[bus] != 1) { vm_bus[bus] = row[OPFG_VG]; vgens[bus]++; }
        }
        G->vm_bus_host = vm_bus;
        G->gen_q_share_host.resize(ng);
        for (int gI = 0; gI < ng; ++gI) {
            const int bus = G->gen_bus_host[gI];
            G->gen_q_share_host[gI] = vgens[bus] ? 1.0 / vgens[bus] : 0.0;
        }
        // branches
        std::vector<BranchHost> active;
        std::vector<double> br_param(6 * (size_t)nbr);
        std::vector<int> br_f(nbr), br_t(nbr);
        for (int l = 0; l < nbr; ++l) {
            const double* row = desc->branch + (size_t)l * desc->branch_cols;
            BranchHost bh;
            bh.f = (int)row[OPFG_F_BUS]; bh.t = (int)row[OPFG_T_BUS];
            if (bh.f < 0 || bh.f >= nb || bh.t < 0 || bh.t >= nb) { delete G; return fail("branch %d has invalid bus", l); }
            bh.r = row[OPFG_BR_R]; bh.x = row[OPFG_BR_X]; bh.b = row[OPFG_BR_B];
            bh.g = desc->branch_cols > OPFG_BR_G ? row[OPFG_BR_G] : 0.0;
            bh.tap = row[OPFG_TAP]; bh.shift_deg = row[OPFG_SHIFT];
            br_f[l] = bh.f; br_t[l] = bh.t;
            double* p = &br_param[6 * (size_t)l];
            const bool on = row[OPFG_BR_STATUS] != 0.0;
            p[0] = bh.r; p[1] = bh.x; p[2] = bh.b; p[3] = bh.g; p[4] = bh.tap; p[5] = bh.shift_deg * M_PI / 180.0;
            if (on) active.push_back(bh);
            else { p[0] = 1e300; p[1] = 0; p[2] = 0; p[3] = 0; }   // open branch: zero admittance
        }
        G->br_f_host = br_f; G->br_t_host = br_t; G->type_host = type;
        G->br_on_host.resize(nbr); G->br_tap_host.resize(nbr);
        for (int l = 0; l < nbr; ++l) {
            G->br_on_host[l] = desc->branch[(size_t)l * desc->branch_cols + OPFG_BR_STATUS] != 0.0;
            G->br_tap_host[l] = desc->branch[(size_t)l * desc->branch_cols + OPFG_TAP];
        }
        // map active branches back to ppc rows for Ybus contributions
        std::vector<int> active_row;
        for (int l = 0; l < nbr; ++l)
            if (desc->branch[(size_t)l * desc->branch_cols + OPFG_BR_STATUS] != 0.0) active_row.push_back(l);

        int T = desc->threads_per_env;
        Symbolic& s = G->sym;
        // pf_kernel 1 keeps the CTA-per-environment kernel (and its level-minimising ordering)
        const int pf_kernel = desc->pf_kernel;
        G->pf_kernel = pf_kernel;
        const bool want_lanes = pf_kernel == 2;     // measured slower than the CTA kernels on B200 (DESIGN.md): opt-in
        if (desc->ordering < 0 || desc->ordering > 3) { delete G; return fail("unknown ordering %d", desc->ordering); }
        // a radial grid has a fill-free (leaf-first) order, which is what the fused kernel needs; rooting every
        // tree at its centre makes its level chain the shortest such an order has
        const bool centre_rooted = desc->ordering == 0 && pf_kernel != 1 && pf_kernel != 2 && is_forest(nb, type, active);
        const int ordering = centre_rooted ? 4 : ((desc->ordering == 0 && want_lanes) ? 3 : desc->ordering);
        analyse(nb, type, active, ordering, T > 0 ? T : 32, s, centre_rooted ? TREE_LANES : 0);
        if (T <= 0) T = s.n_blocks <= 1000 ? 64 : 128;   // measured: 64 on the MV grids (~450 blocks), 128 on HV (~1900)
        for (size_t c = 0; c < s.yc_branch.size(); ++c)
            if (s.yc_role[c] != 4) s.yc_branch[c] = active_row[s.yc_branch[c]];

        GridDev& d = G->d;
        d.nb = nb; d.n = s.n; d.n_levels = s.n_levels; d.n_blocks = s.n_blocks; d.n_fill = (int)s.fill_ids.size();
        d.nnz_y = (int)s.y_col.size(); d.nbr = nbr; d.ng = ng; d.n_ref = n_ref; d.threads = T;
        d.base_mva = base; d.tol = desc->tol_pu; d.max_iter = desc->max_iter; d.init_dc = desc->init_dc;
        std::vector<unsigned char> type_int(nb);
        std::vector<double> vm0(nb), va0(nb);
        for (int i = 0; i < nb; ++i) {
            const int bus = s.bus_of_int[i];
            type_int[i] = (unsigned char)type[bus];
            vm0[i] = vm_bus[bus];
            va0[i] = type[bus] == 3 ? va_ref[bus] : (desc->init_dc ? 0.0 : va_ref[bus]);
        }
        G->tab_reserve(4096 + 16 * (size_t)nb * 8 + 8 * (s.dp_l.size() + s.off_tgt.size() + 1) +
                       4 * (s.op_l.size() + s.up_w.size() + s.fill_ids.size()) + 24 * s.y_col.size() +
                       8 * (size_t)s.n_blocks + 16 * (size_t)s.n_levels + 64 * 32);
        d.bus_of_int = G->tab(s.bus_of_int); d.int_of_bus = G->up(s.int_of_bus);
        d.type_int = G->tab(type_int);
        d.level_ptr = G->tab(s.level_ptr); d.fill_ids = G->tab(s.fill_ids);
        if (s.n_blocks >= 65535 || nb >= 65535) { delete G; return fail("grid too large for 16-bit schedule ids (%d blocks)", s.n_blocks); }
        {   // pack the schedule into 16-bit ids (halves the L1 footprint of the shared tables)
            // ---- storage slots of the blocks (meshed grids) ----
            // A block id names a 2x2 block of the filled Jacobian; the kernel addresses shared memory by SLOT.
            // A fill block does not exist before the off-diagonal item that forms it runs (level of its
            // pivot), and an L~ block is dead once the last item that gathers with it has run (at the latest
            // the level of its row: the right-hand side is carried along, the backward sweep reads W only).
            // So a fill block born in level l takes the slot of a block last read in a level < l (the
            // barrier between two levels orders the last read before the first write): 1 899 blocks ->
            // 1 449 slots on the 372-bus grid, 75.7 -> 61.3 KB per environment -- a THIRD environment per SM.
            // Only addresses change: every sum keeps its operands and its order (same bits).
            std::vector<int> slot(s.n_blocks);
            for (int b = 0; b < s.n_blocks; ++b) slot[b] = b;
            std::vector<char> is_fill(s.n_blocks, 0);
            for (int f : s.fill_ids) is_fill[f] = 1;
            int n_slots = s.n_blocks;
            const bool share_slots = (getenv("OPFG_SHARE_SLOTS") ? atoi(getenv("OPFG_SHARE_SLOTS")) != 0 : true) &&
                                     !s.fill_ids.empty();
            if (share_slots) {
                const int NEVER = 1 << 30;
                std::vector<int> level_of(s.n, 0), last(s.n_blocks, -1), born(s.n_blocks, -1);
                for (int l = 0; l < s.n_levels; ++l)
                    for (int k = s.level_ptr[l]; k < s.level_ptr[l + 1]; ++k) level_of[k] = l;
                auto read_at = [&](int b, int l) { if (last[b] < l) last[b] = l; };
                // a diagonal slot holds D_k (with its eager partial sums), then D_k^-1 until the U blocks of row k are
                // scaled: dead after level(k) as well (t_k lives in the right-hand side)
                for (int k = 0; k < s.n; ++k) {
                    read_at(k, level_of[k]);
                    for (int p = s.dp_ptr[k]; p < s.dp_ptr[k + 1]; ++p) { read_at(s.dp_l[p], level_of[k]); read_at(s.dp_w[p], level_of[k]); }
                }
                for (int l = 0; l < s.n_levels; ++l)
                    for (int item = s.off_ptr[l]; item < s.off_ptr[l + 1]; ++item) {
                        born[s.off_tgt[item]] = l;
                        read_at(s.off_tgt[item], l);
                        if (s.off_piv[item] >= 0) read_at(s.off_piv[item], l);
                        for (int p = s.op_ptr[item]; p < s.op_ptr[item + 1]; ++p) { read_at(s.op_l[p], l); read_at(s.op_w[p], l); }
                    }
                for (int w : s.up_w) last[w] = NEVER;                       // backward sweep
                bool ok = true;
                for (int f : s.fill_ids) ok = ok && born[f] >= 0 && f >= s.n;
                if (ok) {
                    int next = s.n;                                          // diagonals keep slot == pivot
                    for (int b = s.n; b < s.n_blocks; ++b) if (!is_fill[b]) slot[b] = next++;   // written by the Jacobian pass
                    std::vector<std::vector<int>> births(s.n_levels), deaths(s.n_levels);
                    for (int b = 0; b < s.n_blocks; ++b) {
                        if (is_fill[b]) births[born[b]].push_back(b);
                        if (last[b] >= 0 && last[b] < s.n_levels) deaths[last[b]].push_back(b);
                    }
                    std::vector<int> pool;
                    for (int l = 0; l < s.n_levels; ++l) {
                        for (int b : births[l]) {
                            if (!pool.empty()) { slot[b] = pool.back(); pool.pop_back(); }
                            else slot[b] = next++;
                        }
                        for (int b : deaths[l]) pool.push_back(slot[b]);
                    }
                    n_slots = next;
                    // safety net: within one level no item may read a slot another item of that level writes
                    std::vector<int> written_in(n_slots, -1);
                    for (int l = 0; l < s.n_levels && ok; ++l) {
                        for (int item = s.off_ptr[l]; item < s.off_ptr[l + 1]; ++item) written_in[slot[s.off_tgt[item]]] = l;
                        for (int item = s.off_ptr[l]; item < s.off_ptr[l + 1] && ok; ++item)
                            for (int p = s.op_ptr[item]; p < s.op_ptr[item + 1]; ++p)
                                if (written_in[slot[s.op_l[p]]] == l || written_in[slot[s.op_w[p]]] == l) ok = false;
                        for (int k = s.level_ptr[l]; k < s.level_ptr[l + 1] && ok; ++k) if (written_in[k] == l) ok = false;   // own diagonal
                        for (int i = s.eg_ptr[l]; i < s.eg_ptr[l + 1] && ok; ++i) if (written_in[s.eg_k[i]] == l) ok = false;  // eager targets
                        for (int item = s.off_ptr[l]; item < s.off_ptr[l + 1] && ok; ++item)
                            if (s.off_piv[item] >= 0 && written_in[s.off_piv[item]] == l) ok = false;                         // D^-1 of the scale phase
                        for (int k = s.level_ptr[l]; k < s.level_ptr[l + 1] && ok; ++k)   // next level's gathers vs this level's writes: other phase, but
                            for (int p = s.dp_ptr[k]; p < s.dp_ptr[k + 1]; ++p)          // an operand must not have been overwritten in ITS level either
                                if (written_in[slot[s.dp_l[p]]] == l || written_in[slot[s.dp_w[p]]] == l) ok = false;
                    }
                    if (!ok) { for (int b = 0; b < s.n_blocks; ++b) slot[b] = b; n_slots = s.n_blocks; }
                }
            }
            G->n_blocks_sym = s.n_blocks;
            d.n_blocks = n_slots;
            std::vector<U2> dp(s.dp_l.size()), hdr(s.off_tgt.size() + 1);
            std::vector<uint32_t> op(s.op_l.size()), upk(s.up_w.size());
            std::vector<U2> ym(s.y_col.size());
            for (size_t i = 0; i < dp.size(); ++i) dp[i] = U2{(uint32_t)slot[s.dp_l[i]] | ((uint32_t)slot[s.dp_w[i]] << 16), (uint32_t)s.dp_m[i]};
            // bit 31 of the pair pointer: the target is a fill block -- it starts from zero instead of a stored value
            for (size_t i = 0; i < s.off_tgt.size(); ++i)
                hdr[i] = U2{(uint32_t)slot[s.off_tgt[i]] | ((uint32_t)(s.off_piv[i] + 1) << 16),
                            (uint32_t)s.op_ptr[i] | (is_fill[s.off_tgt[i]] ? 0x80000000u : 0u)};
            hdr[s.off_tgt.size()] = U2{0u, (uint32_t)s.op_l.size()};
            for (size_t i = 0; i < op.size(); ++i) op[i] = (uint32_t)slot[s.op_l[i]] | ((uint32_t)slot[s.op_w[i]] << 16);
            for (size_t i = 0; i < upk.size(); ++i) upk[i] = (uint32_t)slot[s.up_w[i]] | ((uint32_t)s.up_j[i] << 16);
            for (int r = 0; r < nb; ++r)
                for (int e = s.y_ptr[r]; e < s.y_ptr[r + 1]; ++e)
                    ym[e] = U2{(uint32_t)s.y_col[e] | ((uint32_t)((s.y_blk[e] < 0 ? -1 : slot[s.y_blk[e]]) + 1) << 16), (uint32_t)r};
            d.nnz_y_nonref = s.y_ptr[s.n];
            // Eager gather pays where few environments fit an SM and the phase latency is exposed
            // (meshed 372-bus grid: -7 %); with ten resident environments the kernel is bound by
            // shared-memory throughput and the extra partial-sum traffic costs 2 %.
            const bool eager = getenv("OPFG_EAGER_GATHER") ? atoi(getenv("OPFG_EAGER_GATHER")) != 0
                             : pf_smem_doubles(n_slots, s.n, nb, T, 0) * sizeof(double) * 5 > 227 * 1024;   // <= 4 environments beside the tables
            if (!eager) {
                for (int k = 0; k < s.n; ++k) s.dp_own[k] = s.dp_ptr[k];
                s.eg_ptr.assign(s.n_levels + 1, 0);
                s.eg_k.clear(); s.eg_begin.clear(); s.eg_count.clear();
            }
            std::vector<U2> eg(s.eg_k.size());
            for (size_t i = 0; i < eg.size(); ++i) {
                if (s.eg_count[i] > 0xffff) throw std::runtime_error("eager gather item with more than 65535 pairs");
                eg[i] = U2{(uint32_t)s.eg_k[i] | ((uint32_t)s.eg_count[i] << 16), (uint32_t)s.eg_begin[i]};
            }
            if (getenv("OPFG_DEBUG_SCHEDULE"))
                for (int l = 0; l < s.n_levels; ++l) {
                    int maxp = 0;
                    for (int k = s.level_ptr[l]; k < s.level_ptr[l + 1]; ++k) maxp = std::max(maxp, s.dp_ptr[k + 1] - s.dp_own[k]);
                    for (int i = s.eg_ptr[l]; i < s.eg_ptr[l + 1]; ++i) maxp = std::max(maxp, s.eg_count[i]);
                    fprintf(stderr, "level %d: own %d eager %d max pairs %d (own max %d) off items %d\n", l,
                            s.level_ptr[l + 1] - s.level_ptr[l], s.eg_ptr[l + 1] - s.eg_ptr[l], maxp,
                            [&] { int m = 0; for (int k = s.level_ptr[l]; k < s.level_ptr[l + 1]; ++k) m = std::max(m, s.dp_ptr[k + 1] - s.dp_ptr[k]); return m; }(),
                            s.off_ptr[l + 1] - s.off_ptr[l]);
                }
            d.dp_ptr = G->tab(s.dp_ptr); d.dp_pack = G->tab(dp);
            d.dp_own = G->tab(s.dp_own); d.eg_ptr = G->tab(s.eg_ptr); d.eg_item = G->tab(eg);
            d.off_ptr = G->tab(s.off_ptr); d.off_hdr = G->tab(hdr); d.op_pack = G->tab(op);
            d.up_ptr = G->tab(s.up_ptr); d.up_pack = G->tab(upk);
            // the Ybus INDEX tables belong to the always-staged part: the row pass reads them in every iteration and
            // every other load of an entry depends on them (their values can be requested ahead by entry number);
            // on the 372-bus grid they are what still fits beside three environments (46 KB + 3 x 61 KB)
            d.y_ptr = G->tab(s.y_ptr); d.y_diag = G->up(s.y_diag); d.y_meta = G->tab(ym);
            d.tab_hot_bytes = (int)((G->tab_used + 15) & ~size_t(15));   // LU schedule + Ybus index tables end here
        }
        d.yc_ptr = G->up(s.yc_ptr); d.yc_branch = G->up(s.yc_branch); d.yc_role = G->up(s.yc_role);
        d.br_param = G->up(br_param); d.bus_ysh = G->up(ysh); d.br_f = G->up(br_f); d.br_t = G->up(br_t);
        d.br_y = (double*)G->up(std::vector<double>(8 * (size_t)nbr, 0.0));
        double* y_val = G->tab(std::vector<double>(2 * s.y_col.size(), 0.0));
        d.y_val = y_val;
        d.tab_warm_bytes = (int)((G->tab_used + 15) & ~size_t(15));   // tables read in every iteration end here
        d.vm0_int = G->tab(vm0); d.va0_int = G->tab(va0);              // start values, q-limits: once per solve

        // DC start: scalar factor of B' on the same schedule + constant part of its rhs
        std::vector<double> dc_val, dc_rhs0(s.n, 0.0);
        bool dc_ok = true;
        factor_dc(s, active, dc_val, dc_ok);
        if (desc->init_dc && !dc_ok) { delete G; return fail("DC matrix B' is singular"); }
        for (const auto& br : active) {
            const double ratio = br.tap == 0.0 ? 1.0 : br.tap;
            const double b = 1.0 / br.x / ratio;
            const double pfinj = b * (-br.shift_deg * M_PI / 180.0);
            const int f = s.int_of_bus[br.f], t = s.int_of_bus[br.t];
            if (f < s.n) dc_rhs0[f] -= pfinj;
            if (t < s.n) dc_rhs0[t] += pfinj;
            // - B'[k, ref] * theta_ref
            if (f < s.n && t >= s.n) dc_rhs0[f] += b * va_ref[br.t];
            if (t < s.n && f >= s.n) dc_rhs0[t] += b * va_ref[br.f];
        }
        for (int k = 0; k < s.n; ++k) dc_rhs0[k] -= ysh[2 * s.bus_of_int[k]];
        d.dc_pre = 0; d.dc_binv_t = nullptr; d.dc_theta0 = nullptr; d.dc_ld = 0;
        // Dense pre-pass for the DC start: theta = B'^-1 (P + rhs0) for ALL environments as one FP64
        // GEMM (k_dc_start).  Inside the persistent kernel the same solve was 2 x levels barrier phases
        // of dependent scalar work: 17 % of the kernel on the 372-bus grid (4.47 -> 3.82 ms with the
        // pre-pass), 11 % on the 122-bus grid (0.14 ms in the kernel against 0.08 ms for the GEMM).
        // B'^-1 is built column by column from the sparse factor of B' on the power-flow schedule.
        if (desc->init_dc && s.n > 0) {
            const int n = s.n, ld = (n + 63) / 64 * 64, kp = (nb + 15) / 16 * 16;   // rows: ppc bus order (coalesced P reads)
            std::vector<double> binv_t((size_t)kp * ld, 0.0), x(n), theta0(n, 0.0);
            auto solve = [&](std::vector<double>& v) {
                for (int l = 0; l < s.n_levels; ++l)
                    for (int k = s.level_ptr[l]; k < s.level_ptr[l + 1]; ++k) {
                        double y = v[k];
                        for (int p = s.dp_ptr[k]; p < s.dp_ptr[k + 1]; ++p) y = std::fma(-dc_val[s.dp_l[p]], v[s.dp_m[p]], y);
                        v[k] = y * dc_val[k];
                    }
                for (int l = s.n_levels - 1; l >= 0; --l)
                    for (int k = s.level_ptr[l]; k < s.level_ptr[l + 1]; ++k) {
                        double xx = v[k];
                        for (int p = s.up_ptr[k]; p < s.up_ptr[k + 1]; ++p) xx = std::fma(-dc_val[s.up_w[p]], v[s.up_j[p]], xx);
                        v[k] = xx;
                    }
            };
            for (int c = 0; c < n; ++c) {
                std::fill(x.begin(), x.end(), 0.0);
                x[c] = 1.0;
                solve(x);                                  // column c of B'^-1
                for (int i = 0; i < n; ++i) binv_t[(size_t)s.bus_of_int[c] * ld + i] = x[i];
            }
            theta0 = dc_rhs0;
            solve(theta0);
            d.dc_binv_t = G->up(binv_t); d.dc_theta0 = G->up(theta0); d.dc_ld = ld; d.dc_pre = 1;
        }
        std::vector<int> lane_qb;
        std::vector<double> lane_qmn, lane_qmx;
        {   // enforce_q_lims tables: one entry per PV bus with an active limit
            std::vector<int> qb;
            std::vector<double> qmn, qmx;
            if (desc->enforce_q_lims && desc->gen_cols > OPFG_QMIN) {
                std::vector<double> mn(nb, 0.0), mx(nb, 0.0);
                std::vector<int> cnt(nb, 0), first(nb, -1);
                for (int gI = 0; gI < ng; ++gI) {
                    const double* row = desc->gen + (size_t)gI * desc->gen_cols;
                    const int bus = (int)row[OPFG_GEN_BUS];
                    if (row[OPFG_GEN_STATUS] <= 0 || type[bus] != 2) continue;
                    // the limits of a bus are pooled into one sum, which equals pandapower's per-generator check
                    // (equal shares of the bus Q) only when every generator of the bus has the same pair
                    if (first[bus] < 0) first[bus] = gI;
                    const double* r0 = desc->gen + (size_t)first[bus] * desc->gen_cols;
                    if (first[bus] != gI && (r0[OPFG_QMIN] != row[OPFG_QMIN] || r0[OPFG_QMAX] != row[OPFG_QMAX])) {
                        delete G;
                        return fail("enforce_q_lims: generator rows %d and %d of PV bus %d (ppc numbering) have different reactive "
                                    "limits (%g, %g) and (%g, %g) MVAr; per-generator limits on one bus are not supported",
                                    first[bus], gI, bus, r0[OPFG_QMIN], r0[OPFG_QMAX], row[OPFG_QMIN], row[OPFG_QMAX]);
                    }
                    // pandapower skips a generator with a zero limit (non_refs = (QMAX != 0) & (QMIN != 0))
                    if (row[OPFG_QMAX] == 0.0 || row[OPFG_QMIN] == 0.0) continue;
                    mn[bus] += row[OPFG_QMIN] / base; mx[bus] += row[OPFG_QMAX] / base; cnt[bus]++;
                }
                for (int b = 0; b < nb; ++b)
                    if (cnt[b]) { qb.push_back(s.int_of_bus[b]); qmn.push_back(mn[b]); qmx.push_back(mx[b]); }
            }
            d.n_qlim = (int)qb.size();
            d.qlim_bus = G->tab(qb); d.qlim_min = G->tab(qmn); d.qlim_max = G->tab(qmx);
            lane_qb = qb; lane_qmn = qmn; lane_qmx = qmx;
        }
        d.tab_base = G->tab_base;
        d.tab_bytes = (int)((G->tab_used + 15) & ~size_t(15));

        // ---- lane-per-environment kernel: row-wise schedule in its own arena ----
        if (want_lanes && nb < 65535 && (int)s.up_w.size() < 65535) {
            LaneSchedule& ls = G->lane;
            build_lane_schedule(s, ls);
            if (ls.max_row <= 255) {
                const int n = s.n;
                std::vector<int> row(4 * (size_t)(n + 1));
                for (int k = 0; k <= n; ++k) {
                    row[4 * k] = s.y_ptr[k]; row[4 * k + 1] = ls.fill_ptr[k];
                    row[4 * k + 2] = ls.el_ptr[k]; row[4 * k + 3] = s.up_ptr[k];
                }
                std::vector<uint32_t> ly(s.y_ptr[n]), el(ls.el_rpos.size()), upd(ls.upd_w.size()), up(s.up_w.size());
                for (size_t e = 0; e < ly.size(); ++e) ly[e] = (uint32_t)s.y_col[e] | ((uint32_t)(ls.y_rpos[e] + 1) << 16);
                for (size_t i = 0; i < el.size(); ++i) el[i] = (uint32_t)ls.el_rpos[i] | ((uint32_t)ls.el_m[i] << 16);
                for (size_t i = 0; i < upd.size(); ++i) upd[i] = (uint32_t)ls.upd_w[i] | ((uint32_t)ls.upd_rpos[i] << 16);
                for (size_t i = 0; i < up.size(); ++i) up[i] = (uint32_t)s.up_j[i] | ((uint32_t)ls.up_rpos[i] << 16);
                std::vector<unsigned char> dpos(ls.diag_pos.begin(), ls.diag_pos.end()), fl(ls.fill_rpos.begin(), ls.fill_rpos.end());
                // the arena is filled through the tab() helper of the main arena: swap the cursors
                char* keep_base = G->tab_base; size_t keep_cap = G->tab_cap, keep_used = G->tab_used;
                G->tab_reserve(1024 + 16 * row.size() / 4 + 4 * (ly.size() + el.size() + ls.el_uptr.size() + upd.size() + up.size()) +
                               dpos.size() + fl.size() + 16 * ly.size() + 21 * (size_t)nb + 20 * lane_qb.size() + 16 * 20);
                G->tab_used = 0;
                d.tab3_base = G->tab_base;
                d.ln_row = G->tab(row); d.ln_y = G->tab(ly); d.ln_diag_pos = G->tab(dpos); d.ln_fill = G->tab(fl);
                d.ln_el = G->tab(el); d.ln_el_uptr = G->tab(ls.el_uptr); d.ln_upd = G->tab(upd); d.ln_up = G->tab(up);
                d.ln_yval = G->tab(std::vector<double>(2 * ly.size(), 0.0));       // filled after the Ybus assembly below
                d.ln_vm0 = G->tab(vm0); d.ln_va0 = G->tab(va0);
                d.ln_bus_of_int = G->tab(s.bus_of_int); d.ln_type = G->tab(type_int);
                d.ln_qbus = G->tab(lane_qb); d.ln_qmin = G->tab(lane_qmn); d.ln_qmax = G->tab(lane_qmx);
                d.tab3_bytes = (int)((G->tab_used + 15) & ~size_t(15));
                G->tab_base = keep_base; G->tab_cap = keep_cap; G->tab_used = keep_used;
                d.ln_max_row = ls.max_row; d.ln_n_up = (int)s.up_w.size();
                G->lanes_ok = true;
            }
        }
        // ---- fused kernel for radial grids: every pivot has at most one later neighbour ----
        d.tr_ok = 0;
        {
            bool forest = pf_kernel != 1 && pf_kernel != 2 && d.n_qlim == 0 && nb < 65535;
            for (int k = 0; k < s.n && forest; ++k) forest = s.up_ptr[k + 1] - s.up_ptr[k] <= 1;
            if (forest) {
                std::vector<int> parent(s.n, -1);
                for (int k = 0; k < s.n; ++k)
                    if (s.up_ptr[k + 1] > s.up_ptr[k]) parent[k] = s.up_j[s.up_ptr[k]];
                std::vector<uint32_t> col(s.y_col.size());
                for (int r = 0; r < nb; ++r)
                    for (int e = s.y_ptr[r]; e < s.y_ptr[r + 1]; ++e) {
                        const int c = s.y_col[e];
                        const uint32_t kind = (r < s.n && c < s.n && c != r) ? (c < r ? 1u : 2u) : 0u;
                        col[e] = (uint32_t)c | (kind << 16);
                    }
                char* keep_base = G->tab_base; size_t keep_cap = G->tab_cap, keep_used = G->tab_used;
                G->tab_reserve(1024 + 4 * (size_t)(3 * nb + s.n_levels + 8) + nb + 4 * col.size() + 16 * col.size() + 40 * (size_t)nb + 16 * 16);
                G->tab_used = 0;
                d.tab4_base = G->tab_base;
                d.tr_y_val = G->tab(std::vector<double>(2 * col.size(), 0.0));      // filled after the Ybus assembly
                d.tr_vm0 = G->tab(vm0); d.tr_va0 = G->tab(va0);
                d.tr_bus_of_int = G->tab(s.bus_of_int); d.tr_level_ptr = G->tab(s.level_ptr);
                d.tr_y_ptr = G->tab(s.y_ptr); d.tr_parent = G->tab(parent);
                d.tr_y_ent = G->tab(col); d.tr_type = G->tab(type_int);
                d.tab4_bytes = (int)((G->tab_used + 15) & ~size_t(15));
                G->tab_base = keep_base; G->tab_cap = keep_cap; G->tab_used = keep_used;
                d.tr_ok = 1;
            }
        }
        G->smem_pf = (pf_smem_doubles(d.n_blocks, s.n, nb, T, d.n_qlim) * sizeof(double) + 31) & ~size_t(31);
        {   // environments per CTA: stage the tables in shared memory when several environments share them
            const size_t budget = 227 * 1024;
            const int cap = std::min(15, 768 / T);    // named barriers 1..15; k_pf_multi is bounded to 768 threads
            // stage everything if at least two environments still fit; else the tables read in every
            // iteration; else only the LU schedule.  (Measured on the 122-bus grid: an 11th environment
            // bought by leaving the start-value tables in global memory is a net loss, 1.46 vs 1.41 ms.)
            auto fit = [&](int bytes) { return (size_t)bytes < budget ? std::min((int)((budget - bytes) / G->smem_pf), cap) : 0; };
            const int sizes[3] = {d.tab_hot_bytes, d.tab_warm_bytes, d.tab_bytes};
            int level = fit(sizes[2]) >= 2 ? 2 : ((fit(sizes[1]) >= 2 && (size_t)sizes[1] * 3 <= budget) ? 1 : 0);
            // with two environments per SM the kernel is latency-bound on 8 warps: a third environment is worth
            // more than staged Ybus tables (372-bus grid, shared slots: 3 x 61 KB + the 34 KB LU schedule)
            if (fit(sizes[level]) <= 2)
                for (int lv = level - 1; lv >= 0; --lv)
                    if (fit(sizes[lv]) > fit(sizes[level])) level = lv;
            if (const char* sv = getenv("OPFG_STAGE")) level = std::max(0, std::min(2, atoi(sv)));
            d.tab_staged_bytes = sizes[level];
            G->stage_level = level;
            int E = fit(sizes[level]);
            if (const char* ev = getenv("OPFG_ENVS_PER_CTA")) E = std::min(atoi(ev), E);   // can only lower it
            if (E < 2) E = 1;
            G->envs_per_cta = E;
            if (getenv("OPFG_DEBUG_SCHEDULE"))
                fprintf(stderr, "blocks %d slots %d: %zu B per environment, tables hot/warm/all %d/%d/%d B, staged level %d, %d environments per CTA\n",
                        G->n_blocks_sym, d.n_blocks, G->smem_pf, sizes[0], sizes[1], sizes[2], level, E);
        }
        G->smem_score = score_smem_doubles(nb, nbr, T) * sizeof(double);
        if (G->smem_pf > 227 * 1024) { delete G; return fail("grid needs %zu B shared memory per environment (> 227 KB)", G->smem_pf); }

        // kernel 1a: branch admittances and Ybus values, computed on the device
#ifdef OPFG_HOSTSIM
        for (int l = 0; l < nbr; ++l) branch_admittance(d.br_param + 6 * (size_t)l, d.br_y + 8 * (size_t)l);
        for (int e = 0; e < d.nnz_y; ++e) ybus_entry(d, d.br_y, e, y_val + 2 * (size_t)e);
#else
        k_branch_y<<<(nbr + 127) / 128, 128>>>(d);
        k_ybus<<<(d.nnz_y + 127) / 128, 128>>>(d, y_val);
        g_launches += 2;
        cudaError_t e = cudaDeviceSynchronize();
        if (e != cudaSuccess) { delete G; return fail("Ybus assembly failed: %s", cudaGetErrorString(e)); }
#endif
        if (d.tr_ok) {
            const size_t ybytes = sizeof(double) * 2 * s.y_col.size();
            G->tree_env_doubles = tree_smem_doubles(s.n, nb);
#ifdef OPFG_HOSTSIM
            memcpy(const_cast<double*>(d.tr_y_val), y_val, ybytes);
#else
            cudaMemcpy(const_cast<double*>(d.tr_y_val), y_val, ybytes, cudaMemcpyDeviceToDevice);
            // lanes per environment: narrow levels (one pivot per feeder) leave wider groups idle; the
            // environments that fit shared memory decide how many warps an SM gets
            constexpr int T = TREE_LANES;
            const size_t budget = 227 * 1024, per_env = G->tree_env_doubles * sizeof(double);
            int E = (size_t)d.tab4_bytes < budget ? (int)((budget - d.tab4_bytes) / per_env) : 0;
            E = std::min(E, 32);                       // the kernel's launch bounds (512 threads)
            if (const char* ev = getenv("OPFG_TREE_ENVS")) E = std::min(E, atoi(ev));
            E -= E % (32 / T);                         // whole warps
            if (E < 32 / T) d.tr_ok = 0;
            G->tree_T = T; G->tree_E = E;
            G->tree_smem = d.tab4_bytes + (size_t)E * per_env;
            int dev = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&G->n_sm, cudaDevAttrMultiProcessorCount, dev);
#endif
        }
        if (G->lanes_ok) {
            const size_t ybytes = sizeof(double) * 2 * (size_t)s.y_ptr[s.n];
#ifdef OPFG_HOSTSIM
            memcpy(const_cast<double*>(d.ln_yval), y_val, ybytes);
            G->lane_warp_doubles = lane_scratch_doubles(nb, s.n, d.ln_n_up, s.y_ptr[s.n]);
            G->lane_scratch = (double*)dev_alloc(sizeof(double) * (G->lane_warp_doubles + 4 * (size_t)d.ln_max_row));
            if (!G->lane_scratch) { delete G; return fail("lane scratch allocation failed"); }
            G->allocs.push_back(G->lane_scratch);
#else
            cudaMemcpy(const_cast<double*>(d.ln_yval), y_val, ybytes, cudaMemcpyDeviceToDevice);
            int dev = 0;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&G->n_sm, cudaDevAttrMultiProcessorCount, dev);
            // launch shape: W warps per CTA, one CTA per SM; shared memory = tables (if they fit) + W row buffers
            const size_t rb_bytes = sizeof(double) * 4 * (size_t)d.ln_max_row * 32;
            const size_t budget = 227 * 1024;
            int W = 12;
            const bool staged = (size_t)d.tab3_bytes + rb_bytes <= budget;
            const size_t tabs = staged ? (size_t)d.tab3_bytes : 0;
            while (W > 1 && tabs + W * rb_bytes > budget) --W;
            if (tabs + W * rb_bytes > budget) G->lanes_ok = false;     // one row buffer does not fit: CTA kernel
            else {
                G->lane_warps_per_cta = W; G->lane_stage = staged; G->lane_ctas = G->n_sm;
                G->lane_smem = tabs + W * rb_bytes;
                G->lane_warp_doubles = lane_scratch_doubles(nb, s.n, d.ln_n_up, s.y_ptr[s.n]) * 32;
                const size_t bytes = sizeof(double) * G->lane_warp_doubles * (size_t)W * G->lane_ctas;
                void* p = nullptr;
                if (cudaMalloc(&p, bytes) != cudaSuccess) { cudaGetLastError(); G->lanes_ok = false; }
                else { G->lane_scratch = (double*)p; G->allocs.push_back(p); }
            }
#endif
        }
        *out = G;
        return 0;
    } catch (const std::exception& ex) {
        return fail("opfg_grid_create: %s", ex.what());
    }
}

void opfg_grid_destroy(OpfgGrid* grid) { delete grid; }

static void check_ref_vm(const OpfgAssemblyDesc* a, int nb) {
    for (int b = 0; b < nb; ++b) {
        const int r = a->bus_vm_ref[b];
        if (r != OPFG_NO_REF && (r >= a->n_state || -r - 1 >= a->n_const))
            throw std::runtime_error("reference out of range in bus_vm_ref");
    }
}

int opfg_set_assembly(OpfgGrid* G, const OpfgAssemblyDesc* a) {
    if (!G || !a) return fail("null argument");
    try {
        GridDev& d = G->d;
        d.n_state = a->n_state; d.n_const = a->n_const; d.n_act = a->n_act; d.n_inj = a->n_inj;
        d.act_diff_step = a->act_diff_step;
        d.consts = G->up(a->consts, a->n_const);
        G->consts_host.assign(a->consts, a->consts + a->n_const);
        {
            std::vector<double> rev(G->consts_host.rbegin(), G->consts_host.rend());
            d.consts_end = G->up(rev) + a->n_const;
        }
        auto check_ref = [&](const int* r, int n, const char* what) {
            for (int i = 0; i < n; ++i)
                if (r[i] >= a->n_state || -r[i] - 1 >= a->n_const) throw std::runtime_error(std::string("reference out of range in ") + what);
        };
        check_ref(a->act_lo, a->n_act, "act_lo"); check_ref(a->act_hi, a->n_act, "act_hi");
        check_ref(a->act_div, a->n_act, "act_div");
        check_ref(a->inj_p, a->n_inj, "inj_p"); check_ref(a->inj_q, a->n_inj, "inj_q"); check_ref(a->inj_coef, a->n_inj, "inj_coef");
        for (int i = 0; i < a->n_act; ++i)
            if (a->act_slot[i] < 0 || a->act_slot[i] >= a->n_state) throw std::runtime_error("act_slot out of range");
        G->act_ref_max = -1;
        for (int i = 0; i < a->n_act; ++i) {
            G->act_ref_max = std::max({G->act_ref_max, a->act_slot[i], a->act_lo[i], a->act_hi[i], a->act_div[i]});
            if (a->act_clamp_lo) G->act_ref_max = std::max({G->act_ref_max, a->act_clamp_lo[i], a->act_clamp_hi[i]});
        }
        d.act_slot = G->up(a->act_slot, a->n_act);
        d.act_lo = G->up(a->act_lo, a->n_act); d.act_hi = G->up(a->act_hi, a->n_act);
        d.act_div = G->up(a->act_div, a->n_act); d.act_kind = G->up(a->act_kind, a->n_act);
        d.act_clamp_lo = a->act_clamp_lo ? G->up(a->act_clamp_lo, a->n_act) : nullptr;
        d.act_clamp_hi = a->act_clamp_hi ? G->up(a->act_clamp_hi, a->n_act) : nullptr;
        // CSR by bus, list order preserved (deterministic summation order)
        std::vector<int> ptr(d.nb + 1, 0), p(a->n_inj), q(a->n_inj), c(a->n_inj);
        for (int e = 0; e < a->n_inj; ++e) {
            if (a->inj_bus[e] < 0 || a->inj_bus[e] >= d.nb) throw std::runtime_error("injection on invalid bus");
            ptr[a->inj_bus[e] + 1]++;
        }
        for (int b = 0; b < d.nb; ++b) ptr[b + 1] += ptr[b];
        std::vector<int> fill(ptr.begin(), ptr.end() - 1);
        for (int e = 0; e < a->n_inj; ++e) {
            const int at = fill[a->inj_bus[e]]++;
            p[at] = a->inj_p[e]; q[at] = a->inj_q[e]; c[at] = a->inj_coef[e];
        }
        d.inj_ptr = G->up(ptr); d.inj_p = G->up(p); d.inj_q = G->up(q); d.inj_coef = G->up(c);
        std::vector<int> order(d.nb);
        for (int b = 0; b < d.nb; ++b) order[b] = b;
        std::stable_sort(order.begin(), order.end(), [&](int a_, int b_) { return ptr[a_ + 1] - ptr[a_] > ptr[b_ + 1] - ptr[b_]; });
        d.inj_order = G->up(order);
        d.vm_from_state = 0; d.bus_vm_ref = nullptr; d.vm0_bus = nullptr;
        if (a->bus_vm_ref) {
            check_ref_vm(a, d.nb);
            std::vector<double> vm0_bus(d.nb);
            for (int b = 0; b < d.nb; ++b) vm0_bus[b] = G->vm_bus_host[b];
            d.bus_vm_ref = G->up(a->bus_vm_ref, d.nb); d.vm0_bus = G->up(vm0_bus);
            d.vm_from_state = 1;
        }
        G->has_assembly = true;
        return 0;
    } catch (const std::exception& ex) {
        return fail("opfg_set_assembly: %s", ex.what());
    }
}

int opfg_set_dynamic_branches(OpfgGrid* G, const OpfgDynBranchDesc* dd) {
    if (!G || !dd) return fail("null argument");
    if (!G->has_assembly) return fail("call opfg_set_assembly first (it defines the state layout)");
    try {
        GridDev& d = G->d;
        std::vector<int> of(d.nbr, -1);
        for (int i = 0; i < dd->n_dyn; ++i) {
            const int br = dd->branch[i];
            if (br < 0 || br >= d.nbr) throw std::runtime_error("dynamic branch out of range");
            if (of[br] >= 0) throw std::runtime_error("branch listed twice");
            of[br] = i;
            for (const int* r : {dd->tap_pos + i, dd->in_service + i, dd->closed_from ? dd->closed_from + i : nullptr,
                                 dd->closed_to ? dd->closed_to + i : nullptr})
                if (r && (*r >= d.n_state || -*r - 1 >= d.n_const)) throw std::runtime_error("reference out of range");
        }
        // optional arrays: no switches (the in-service reference stands in: same value, "closed" wherever the
        // branch is in service at all would be wrong for a cleared cell, so point at a constant that is not 0)
        std::vector<int> cf(dd->n_dyn), ct(dd->n_dyn), flags(dd->n_dyn, 0);
        std::vector<double> lv_scale(dd->n_dyn, 1.0);
        int one_ref = 0;
        {
            std::vector<double> cs(d.n_const);
            dev_get(cs.data(), d.consts, sizeof(double) * d.n_const);
            int found = -1;
            for (int c = 0; c < d.n_const && found < 0; ++c) if (cs[c] == 1.0) found = c;
            if (found < 0 && (!dd->closed_from || !dd->closed_to)) throw std::runtime_error("constant table holds no 1.0");
            one_ref = -found - 1;
        }
        for (int i = 0; i < dd->n_dyn; ++i) {
            cf[i] = dd->closed_from ? dd->closed_from[i] : one_ref;
            ct[i] = dd->closed_to ? dd->closed_to[i] : one_ref;
            flags[i] = dd->flags ? dd->flags[i] : 0;
            if (flags[i] & OPFG_DYN_TAP_LV) {
                // the ppc row carries the parameters at the static tap t0 = ratio_neutral / ratio_static
                const double ratio_static = G->br_tap_host[dd->branch[i]] == 0.0 ? 1.0 : G->br_tap_host[dd->branch[i]];
                const double t0 = dd->ratio_neutral[i] / ratio_static;
                lv_scale[i] = 1.0 / (t0 * t0);
            }
        }
        d.n_dyn = dd->n_dyn;
        d.dyn_branch = G->up(dd->branch, dd->n_dyn);
        d.dyn_of_branch = G->up(of);
        d.dyn_tap_ref = G->up(dd->tap_pos, dd->n_dyn);
        d.dyn_svc_ref = G->up(dd->in_service, dd->n_dyn);
        d.dyn_neutral = G->up(dd->tap_neutral, dd->n_dyn);
        d.dyn_step = G->up(dd->tap_step_percent, dd->n_dyn);
        d.dyn_ratio0 = G->up(dd->ratio_neutral, dd->n_dyn);
        d.dyn_cf_ref = G->up(cf); d.dyn_ct_ref = G->up(ct); d.dyn_flags = G->up(flags); d.dyn_lv_scale = G->up(lv_scale);
        // Islands.  Spanning forest of the static grid from the slack buses, branches WITHOUT an in-service
        // cell first: a dynamic branch that still becomes a tree edge is "critical" -- only when one of those
        // is out can an environment lose buses, and only then does kernel 1 walk the grid (open ties that
        // merely close loops never trigger the walk).
        d.isl = 0; d.dyn_crit = nullptr; d.isl_ptr = d.isl_adj = d.isl_br = nullptr; G->n_crit = 0;
        bool any_switchable = false;
        std::vector<unsigned char> switchable(d.nbr, 0);
        for (int i = 0; i < dd->n_dyn; ++i) {
            // references to constants that are not 0 mean "always in service / closed"
            bool fixed_on = true;
            for (int r : {dd->in_service[i], cf[i], ct[i]}) {
                if (r >= 0) { fixed_on = false; continue; }
                double c;
                dev_get(&c, d.consts + (-r - 1), sizeof(double));
                fixed_on = fixed_on && c != 0.0;
            }
            if (!fixed_on && G->br_on_host[dd->branch[i]]) { switchable[dd->branch[i]] = 1; any_switchable = true; }
        }
        if (any_switchable) {
            const int nb = d.nb, nbr = d.nbr;
            std::vector<int> ptr(nb + 1, 0), adj, brs;
            for (int l = 0; l < nbr; ++l)
                if (G->br_on_host[l] && G->br_f_host[l] != G->br_t_host[l]) { ptr[G->br_f_host[l] + 1]++; ptr[G->br_t_host[l] + 1]++; }
            for (int b = 0; b < nb; ++b) ptr[b + 1] += ptr[b];
            adj.resize(ptr[nb]); brs.resize(ptr[nb]);
            std::vector<int> fillp(ptr.begin(), ptr.end() - 1);
            // switchable[l]: 1 = normally in service, 2 = normally open (hint): the forest grows through the former first,
            // so that ties which merely close loops do not become "critical"
            for (int i = 0; i < dd->n_dyn; ++i)
                if (switchable[dd->branch[i]] && (flags[i] & OPFG_DYN_NORMALLY_OPEN)) switchable[dd->branch[i]] = 2;
            for (int pass = 0; pass < 3; ++pass)          // fixed branches first: the walk meets them first, too
                for (int l = 0; l < nbr; ++l) {
                    if (!G->br_on_host[l] || G->br_f_host[l] == G->br_t_host[l] || (int)switchable[l] != pass) continue;
                    const int f = G->br_f_host[l], t = G->br_t_host[l];
                    adj[fillp[f]] = t; brs[fillp[f]++] = l;
                    adj[fillp[t]] = f; brs[fillp[t]++] = l;
                }
            // forest: breadth-first over the fixed branches, then extended through switchable ones
            std::vector<char> seen(nb, 0);
            std::vector<unsigned char> crit(dd->n_dyn, 0);
            std::vector<int> queue;
            for (int b = 0; b < nb; ++b) if (G->type_host[b] == 3) { seen[b] = 1; queue.push_back(b); }
            size_t head = 0;
            for (;;) {
                for (; head < queue.size(); ++head) {
                    const int a = queue[head];
                    for (int e = ptr[a]; e < ptr[a + 1]; ++e)
                        if (!switchable[brs[e]] && !seen[adj[e]]) { seen[adj[e]] = 1; queue.push_back(adj[e]); }
                }
                bool grown = false;                        // one switchable edge out of the reached set, then go on
                for (int kind = 1; kind <= 2 && !grown; ++kind)
                    for (size_t q = 0; q < queue.size() && !grown; ++q) {
                        const int a = queue[q];
                        for (int e = ptr[a]; e < ptr[a + 1] && !grown; ++e)
                            if (switchable[brs[e]] == kind && !seen[adj[e]]) {
                                seen[adj[e]] = 1; queue.push_back(adj[e]);
                                crit[of[brs[e]]] = 1; grown = true;
                            }
                    }
                if (!grown) break;
            }
            bool any_crit = false;
            for (unsigned char c : crit) { any_crit |= c != 0; G->n_crit += c != 0; }
            if (any_crit) {
                d.dyn_crit = G->up(crit); d.isl_ptr = G->up(ptr); d.isl_adj = G->up(adj); d.isl_br = G->up(brs);
                d.isl = 1;
                if (!d.vm_from_state) {                    // kernel 1 writes every start |V|: the mark of a dropped bus is 0
                    std::vector<int> no_ref(nb, OPFG_NO_REF);
                    d.bus_vm_ref = G->up(no_ref); d.vm0_bus = G->up(G->vm_bus_host);
                    d.vm_from_state = 1;
                }
            }
        }
        return 0;
    } catch (const std::exception& ex) {
        return fail("opfg_set_dynamic_branches: %s", ex.what());
    }
}

int opfg_set_scoring(OpfgGrid* G, const OpfgScoringDesc* sc) {
    if (!G || !sc) return fail("null argument");
    if (!G->has_assembly) return fail("call opfg_set_assembly first (it defines the state layout)");
    try {
        GridDev& d = G->d;
        const int nbr = d.nbr, ng = d.ng;
        const int n_el = sc->n_constraints ? sc->con_ptr[sc->n_constraints] : 0;
        {
            const size_t cap = 8192 + 16 * (size_t)sc->n_pp_bus + 96 * (size_t)nbr + 32 * (size_t)ng + 48 * (size_t)n_el +
                               64 * (size_t)sc->n_constraints + 64 * (size_t)sc->n_poly + 32 * (size_t)sc->n_pwl * (sc->n_pwl_seg + 1) +
                               8 * (size_t)sc->n_obs + 8 * G->consts_host.size() + 16 * (size_t)d.nb +
                               (sc->n_trafo3w > 0 ? 32 + 8 * (size_t)sc->n_trafo3w : 0);
            G->tab2_base = (char*)dev_alloc(cap);
            if (!G->tab2_base) throw std::runtime_error("device allocation failed");
            G->allocs.push_back(G->tab2_base);
            G->tab2_cap = cap; G->tab2_used = 0;
        }
        d.n_pp_bus = sc->n_pp_bus;
        d.pp_lookup = G->tab2(sc->pp_bus_lookup, sc->n_pp_bus);
        d.res_vm_slot = sc->res_bus_vm_slot; d.res_va_slot = sc->res_bus_va_slot;
        d.br_loading_slot = G->tab2(sc->branch_loading_slot, nbr);
        d.br_flow_slot = G->tab2(sc->branch_flow_slot, nbr);
        d.rate_f = G->tab2(sc->rate_f, nbr); d.rate_t = G->tab2(sc->rate_t, nbr);
        d.n_t3 = 0; d.t3_row_slot = d.t3_loading_slot = nullptr;
        if (sc->n_trafo3w < 0) throw std::runtime_error("n_trafo3w < 0");
        if (sc->n_trafo3w > 0) {
            const int n3 = sc->n_trafo3w;
            if (!sc->trafo3w_row_slot || !sc->trafo3w_loading_slot) throw std::runtime_error("trafo3w tables missing");
            for (int k = 0; k < n3; ++k) {
                const int rs = sc->trafo3w_row_slot[k], ls = sc->trafo3w_loading_slot[k];
                if (rs < sc->n_inputs || rs + 3 > d.n_state || ls < sc->n_inputs || ls >= d.n_state)
                    throw std::runtime_error("trafo3w result slot out of range");
            }
            d.n_t3 = n3;
            d.t3_row_slot = G->tab2(sc->trafo3w_row_slot, n3);
            d.t3_loading_slot = G->tab2(sc->trafo3w_loading_slot, n3);
        }
        d.gen_bus = G->tab2(G->gen_bus_host);
        d.gen_q_share = G->tab2(G->gen_q_share_host);
        d.gen_p_slot = G->tab2(sc->gen_p_slot, ng); d.gen_q_slot = G->tab2(sc->gen_q_slot, ng);
        d.n_con = sc->n_constraints;
        d.con_ptr = G->tab2(sc->con_ptr, sc->n_constraints + 1);
        d.con_value = G->tab2(sc->con_value, n_el); d.con_value_scale = G->tab2(sc->con_value_scale, n_el);
        d.con_min = G->tab2(sc->con_min, n_el); d.con_max = G->tab2(sc->con_max, n_el);
        d.con_bound_mul = G->tab2(sc->con_bound_mul, n_el);
        d.con_autoscale = G->tab2(sc->con_autoscale, d.n_con); d.con_worst = G->tab2(sc->con_worst_case, d.n_con);
        d.con_pfactor = G->tab2(sc->con_penalty_factor, d.n_con); d.con_ppower = G->tab2(sc->con_penalty_power, d.n_con);
        d.con_pcount = G->tab2(sc->con_count_penalty, d.n_con);
        d.n_poly = sc->n_poly; d.n_pwl = sc->n_pwl; d.n_pwl_seg = sc->n_pwl_seg;
        d.poly_p = G->tab2(sc->poly_p, d.n_poly); d.poly_q = G->tab2(sc->poly_q, d.n_poly);
        d.poly_p_mul = G->tab2(sc->poly_p_mul, d.n_poly); d.poly_q_mul = G->tab2(sc->poly_q_mul, d.n_poly);
        d.poly_coef = G->tab2(sc->poly_coef, 6 * (size_t)d.n_poly);
        d.pwl_v = G->tab2(sc->pwl_v, d.n_pwl); d.pwl_v_mul = G->tab2(sc->pwl_v_mul, d.n_pwl);
        d.pwl_seg = G->tab2(sc->pwl_seg, 3 * (size_t)d.n_pwl * d.n_pwl_seg);
        d.reward_kind = sc->reward_kind; d.penalty_weight = sc->penalty_weight;
        d.clip_lo = sc->clip_lo; d.clip_hi = sc->clip_hi;
        d.obj_factor = sc->objective_factor; d.obj_bias = sc->objective_bias;
        d.pen_factor = sc->penalty_factor; d.pen_bias = sc->penalty_bias;
        d.valid_reward = sc->valid_reward; d.invalid_penalty = sc->invalid_penalty;
        d.invalid_obj_share = sc->invalid_objective_share;
        d.n_obs = sc->n_obs;
        d.obs_ref = G->tab2(sc->obs_ref, sc->obs_ptr ? sc->obs_ptr[sc->n_obs] : sc->n_obs);
        G->obs_ref_max = -1;
        for (int i = 0, n = sc->obs_ptr ? sc->obs_ptr[sc->n_obs] : sc->n_obs; i < n; ++i)
            G->obs_ref_max = std::max(G->obs_ref_max, sc->obs_ref[i]);
        d.obs_ptr = sc->obs_ptr ? G->tab2(sc->obs_ptr, sc->n_obs + 1) : nullptr;
        d.n_obs_runs = 0; d.obs_runs = nullptr;
        if (!sc->obs_ptr && sc->n_obs > 0) {      // runs of consecutive state cells (observation keys are whole columns)
            std::vector<int> runs;
            bool ok = true;
            for (int i = 0; i < sc->n_obs && ok;) {
                if (sc->obs_ref[i] < 0) { ok = false; break; }
                int j = i + 1;
                while (j < sc->n_obs && sc->obs_ref[j] == sc->obs_ref[j - 1] + 1) ++j;
                runs.insert(runs.end(), {sc->obs_ref[i], i, j - i});
                i = j;
            }
            if (ok && runs.size() / 3 <= 64 && (int)(runs.size() / 3) * 8 <= sc->n_obs) {
                d.obs_runs = G->up(runs);
                d.n_obs_runs = (int)(runs.size() / 3);
            }
        }
        d.tab2_base = G->tab2_base;
        d.tab2_bytes = (int)((G->tab2_used + 15) & ~size_t(15));
        d.n_inputs = sc->n_inputs;
        if (sc->n_inputs < 0 || sc->n_inputs > d.n_state) throw std::runtime_error("n_inputs out of range");
        int cells = 0;
        if (d.res_vm_slot >= 0) cells += d.n_pp_bus;
        if (d.res_va_slot >= 0) cells += d.n_pp_bus;
        for (int l = 0; l < nbr; ++l) cells += (sc->branch_loading_slot[l] >= 0) + 4 * (sc->branch_flow_slot[l] >= 0);
        for (int gI = 0; gI < ng; ++gI) cells += (sc->gen_p_slot[gI] >= 0) + (sc->gen_q_slot[gI] >= 0);
        cells += sc->n_trafo3w;       // res_trafo3w.loading_percent (its rows' cells are counted with the branches)
        G->n_result_cells = cells;
        G->flops_score = 60.0 * nbr + 30.0 * d.nb + 10.0 * n_el + 14.0 * d.n_poly + 20.0 * d.n_pwl * d.n_pwl_seg + 40.0;
        {   // one warp per environment on small grids: reductions are pure shuffles, no barriers
            int T = (d.nb + nbr <= 600) ? 32 : d.threads;
            if (const char* tv = getenv("OPFG_SCORE_THREADS")) T = atoi(tv);
            G->score_threads = T;
        }
        G->has_scoring = true;
        return 0;
    } catch (const std::exception& ex) {
        return fail("opfg_set_scoring: %s", ex.what());
    }
}

int opfg_grid_info(const OpfgGrid* G, OpfgGridInfo* o) {
    if (!G || !o) return fail("null argument");
    const GridDev& d = G->d;
    memset(o, 0, sizeof *o);
    o->nb = d.nb; o->n_nonref = d.n; o->nnz_y = d.nnz_y; o->n_blocks = G->n_blocks_sym; o->n_fill_blocks = d.n_fill;
    o->n_levels = d.n_levels; o->threads_per_env = d.threads;
    o->smem_bytes_pf = (int)G->smem_pf; o->smem_bytes_score = (int)G->smem_score;
    o->n_state = d.n_state; o->n_const = d.n_const; o->n_act = d.n_act; o->n_obs = d.n_obs; o->n_constraints = d.n_con;
    o->flops_per_iter = G->sym.flops_per_iter; o->lu_flops = G->sym.lu_flops; o->flops_score = G->flops_score;
    // algorithmic HBM bytes of one env step: read action + input state, write results, per-constraint
    // metrics, reward/objective/penalty/cost, flags and the f32 observation (SURVEY.md §8d)
    const int n_in = d.n_state - G->n_result_cells;
    {
        OpfgBatch none{};
        o->pf_kernel_used = use_tree(G, &none) ? 3 : (use_lanes(G, &none) ? 2 : 1);
        o->radial_lanes_per_env = G->tree_T; o->radial_envs_per_cta = G->tree_E;
        o->radial_smem_bytes_per_env = (int)(G->tree_env_doubles * 8);
        o->n_island_critical = G->n_crit;
        o->cta_envs_per_cta = G->envs_per_cta; o->cta_tables_staged = G->stage_level;
        o->score_threads_per_env = G->score_threads;
        o->lane_max_row = d.ln_max_row; o->lane_warps_per_cta = G->lane_warps_per_cta; o->lane_tables_staged = G->lane_stage;
        o->lane_scratch_bytes = 8.0 * (double)G->lane_warp_doubles * std::max(1, G->lane_warps_per_cta * G->lane_ctas);
    }
    o->bytes_per_step = 8.0 * (n_in + d.n_act) + 8.0 * (2.0 * d.nb + G->n_result_cells) + 17.0 * d.n_con + 8.0 * 4 + 5
                        + 4.0 * d.n_obs;
    return 0;
}

int opfg_grid_symbolic(const OpfgGrid* G, int32_t* perm, int32_t* level_ptr) {
    if (!G) return fail("null argument");
    if (perm) for (int k = 0; k < G->sym.n; ++k) perm[k] = G->sym.bus_of_int[k];
    if (level_ptr) for (int l = 0; l <= G->sym.n_levels; ++l) level_ptr[l] = G->sym.level_ptr[l];
    return 0;
}

int opfg_philox_uniform(uint64_t seed, uint64_t first_env, uint64_t stream_id, int64_t n_env, int32_t n_cols,
                        double* out, void* cuda_stream) {
    if (!out || n_env < 0 || n_cols < 0) return fail("bad argument");
    if (n_env == 0 || n_cols == 0) return 0;
    const int pairs = (n_cols + 1) / 2;
#ifdef OPFG_HOSTSIM
    (void)cuda_stream;
    for (int64_t b = 0; b < n_env; ++b)
        for (int pr = 0; pr < pairs; ++pr) {
            double u0, u1;
            philox_two_doubles(seed, first_env + (uint64_t)b, stream_id, (uint32_t)pr, &u0, &u1);
            out[b * n_cols + 2 * pr] = u0;
            if (2 * pr + 1 < n_cols) out[b * n_cols + 2 * pr + 1] = u1;
        }
#else
    const ItemGrid ig = item_grid(n_env, pairs);
    k_philox<<<ig.grid, 256, 0, (cudaStream_t)cuda_stream>>>(seed, first_env, stream_id, n_env, n_cols, out, ig.w_log2);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("philox launch: %s", cudaGetErrorString(e));
#endif
    return 0;
}

int opfg_sample_uniform(uint64_t seed, uint64_t first_env, uint64_t stream_id, int64_t n_env, int32_t n_cols,
                        const int32_t* slots, const double* lo, const double* hi, const double* dv, double* state,
                        int32_t n_state, void* cuda_stream) {
    return opfg_sample_uniform_obs(seed, first_env, stream_id, n_env, n_cols, slots, lo, hi, dv, state, n_state,
                                   nullptr, nullptr, nullptr, 0, cuda_stream);
}

int opfg_sample_uniform_obs(uint64_t seed, uint64_t first_env, uint64_t stream_id, int64_t n_env, int32_t n_cols,
                            const int32_t* slots, const double* lo, const double* hi, const double* dv, double* state,
                            int32_t n_state, const int32_t* obs_pos, float* obs_f32, double* obs_f64, int32_t n_obs,
                            void* cuda_stream) {
    if (!slots || !lo || !hi || !dv || !state || n_env < 0 || n_cols < 0) return fail("bad argument");
    if (obs_pos && ((obs_f32 != nullptr) == (obs_f64 != nullptr) || n_obs <= 0))
        return fail("opfg_sample_uniform_obs: exactly one of obs_f32 / obs_f64, and n_obs > 0");
    if (n_env == 0 || n_cols == 0) return 0;
    const int pairs = (n_cols + 1) / 2;
#ifdef OPFG_HOSTSIM
    (void)cuda_stream;
    for (int64_t b = 0; b < n_env; ++b)
        for (int pr = 0; pr < pairs; ++pr) {
            double u[2];
            philox_two_doubles(seed, first_env + (uint64_t)b, stream_id, (uint32_t)pr, &u[0], &u[1]);
            for (int h = 0; h < 2; ++h) {
                const int j = 2 * pr + h;
                if (j >= n_cols) continue;
                const double v = (lo[j] + (hi[j] - lo[j]) * u[h]) / dv[j];
                state[b * (int64_t)n_state + slots[j]] = v;
                if (obs_pos && obs_pos[j] >= 0) {
                    if (obs_f32) obs_f32[b * (int64_t)n_obs + obs_pos[j]] = (float)v;
                    else obs_f64[b * (int64_t)n_obs + obs_pos[j]] = v;
                }
            }
        }
#else
    const ItemGrid ig = item_grid(n_env, pairs);
    k_sample_uniform<<<ig.grid, 256, 0, (cudaStream_t)cuda_stream>>>(
        seed, first_env, stream_id, n_env, n_cols, slots, lo, hi, dv, state, n_state, ig.w_log2, obs_pos, obs_f32,
        obs_f64, n_obs);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("sample launch: %s", cudaGetErrorString(e));
#endif
    return 0;
}

int opfg_sample_profiles(uint64_t seed, uint64_t first_env, uint64_t stream_id, int64_t n_env, int32_t n_cols,
                         const int32_t* slots, const double* table, int32_t n_steps, const int64_t* step,
                         const double* interp_r, const double* pmin, const double* pmax, double noise_factor,
                         int32_t noise_kind, double* state, int32_t n_state, void* cuda_stream) {
    if (!slots || !table || !step || !pmin || !pmax || !state || n_env < 0 || n_cols < 0 || n_steps <= 0 ||
        noise_kind < 0 || noise_kind > 2)
        return fail("bad argument");
    if (n_env == 0 || n_cols == 0) return 0;
#ifdef OPFG_HOSTSIM
    (void)cuda_stream;
    for (int64_t b = 0; b < n_env; ++b)
        for (int j = 0; j < n_cols; ++j)
            state[b * (int64_t)n_state + slots[j]] = profile_value(seed, first_env + (uint64_t)b, stream_id, j, n_cols, table,
                                                                   n_steps, step[b], interp_r ? interp_r + b : nullptr,
                                                                   pmin, pmax, noise_factor, noise_kind);
#else
    const ItemGrid ig = item_grid(n_env, n_cols);
    k_sample_profiles<<<ig.grid, 256, 0, (cudaStream_t)cuda_stream>>>(
        seed, first_env, stream_id, n_env, n_cols, slots, table, n_steps, step, interp_r, pmin, pmax, noise_factor,
        noise_kind, state, n_state, ig.w_log2);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("profile sampler launch: %s", cudaGetErrorString(e));
#endif
    return 0;
}

int opfg_assemble(const OpfgGrid* G, const OpfgBatch* B, void* stream) {
    if (!G || !B) return fail("null argument");
    if (!G->has_assembly) return fail("opfg_set_assembly was not called");
    if (!B->state || (!B->sbus && !B->actions)) return fail("opfg_assemble needs state and at least one of actions / sbus");
    if (G->d.n_dyn > 0 && B->sbus && (!B->yval || !B->bry)) return fail("grid has dynamic branches: batch needs yval and bry");
    if (G->d.vm_from_state && B->sbus && !B->vm) return fail("grid has per-environment voltage set-points: batch needs vm");
    if (B->n_env <= 0) return 0;
#ifdef OPFG_HOSTSIM
    (void)stream;
    Ctx<1> cx;
    for (int64_t env = 0; env < B->n_env; ++env)
        env_assemble(G->d, cx, B->actions ? B->actions + env * G->d.n_act : nullptr,
                     B->state + env * (int64_t)G->d.n_state, B->sbus ? B->sbus + env * (int64_t)G->d.nb * 2 : nullptr,
                     B->yval ? B->yval + env * (int64_t)G->d.nnz_y * 2 : nullptr,
                     B->bry ? B->bry + env * (int64_t)G->d.n_dyn * 8 : nullptr, B->absolute_actions != 0,
                     B->vm ? B->vm + env * (int64_t)G->d.nb : nullptr);
#else
    k_assemble_warps<<<(unsigned)((B->n_env + 1) / 2), 64, 0, (cudaStream_t)stream>>>(G->d, *B);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("assemble launch: %s", cudaGetErrorString(e));
#endif
    return 0;
}

int opfg_pf_solve(const OpfgGrid* G, const OpfgBatch* B, void* stream) {
    if (!G || !B) return fail("null argument");
    if (!B->sbus || !B->vm || !B->va || !B->converged || !B->iterations) return fail("opfg_pf_solve needs sbus, vm, va, converged, iterations");
    if (B->n_env <= 0) return 0;
#ifdef OPFG_HOSTSIM
    (void)stream;
    Ctx<1> cx;
    std::vector<double> sm(pf_smem_doubles(G->d.n_blocks, G->d.n, G->d.nb, 32, G->d.n_qlim));
    if (G->d.dc_pre) {   // the dense DC pre-pass, as a plain loop
        const GridDev& d = G->d;
        for (int64_t env = 0; env < B->n_env; ++env)
            for (int i = 0; i < d.n; ++i) {
                double acc = 0.0;
                for (int bus = 0; bus < d.nb; ++bus)
                    acc = std::fma(B->sbus[(env * d.nb + bus) * 2], d.dc_binv_t[(size_t)bus * d.dc_ld + i], acc);
                B->va[env * d.nb + d.bus_of_int[i]] = acc + d.dc_theta0[i];
            }
    }
    if (use_tree(G, B)) {
        const GridDev& d = G->d;
        Grp<1> gx;
        std::vector<double> tsm(G->tree_env_doubles);
        const bool dyn = d.n_dyn > 0 && B->yval;
        for (int64_t env = 0; env < B->n_env; ++env)
            env_pf_tree<Grp<1>, true>(d, gx, tsm.data(), B->sbus + env * (int64_t)d.nb * 2,
                        dyn ? B->yval + env * (int64_t)d.nnz_y * 2 : nullptr, B->vm + env * (int64_t)d.nb,
                        B->va + env * (int64_t)d.nb, B->converged + env, B->iterations + env, true);
        return 0;
    }
    if (use_lanes(G, B)) {
        const GridDev& d = G->d;
        const LaneMem<1> s = lane_carve<1>(G->lane_scratch, G->lane_scratch + G->lane_warp_doubles, d.nb, d.n, d.ln_n_up);
        const bool dyn = d.n_dyn > 0 && B->yval;
        for (int64_t env = 0; env < B->n_env; ++env) {
            const double* sb = B->sbus + env * (int64_t)d.nb * 2;
            const double* yv = dyn ? B->yval + env * (int64_t)d.nnz_y * 2 : nullptr;
            double *vm = B->vm + env * (int64_t)d.nb, *va = B->va + env * (int64_t)d.nb;
            if (d.n_qlim > 0 && dyn) lanes_pf_solve<1, true, true>(d, s, sb, yv, vm, va, B->converged + env, B->iterations + env, true);
            else if (d.n_qlim > 0) lanes_pf_solve<1, true, false>(d, s, sb, yv, vm, va, B->converged + env, B->iterations + env, true);
            else if (dyn) lanes_pf_solve<1, false, true>(d, s, sb, yv, vm, va, B->converged + env, B->iterations + env, true);
            else lanes_pf_solve<1, false, false>(d, s, sb, yv, vm, va, B->converged + env, B->iterations + env, true);
        }
        return 0;
    }
    for (int64_t env = 0; env < B->n_env; ++env)
        env_pf_solve(G->d, cx, sm.data(), B->sbus + env * (int64_t)G->d.nb * 2,
                     (G->d.n_dyn > 0 && B->yval) ? B->yval + env * (int64_t)G->d.nnz_y * 2 : nullptr, B->vm + env * (int64_t)G->d.nb,
                     B->va + env * (int64_t)G->d.nb, B->converged + env, B->iterations + env);
#else
    if (G->d.dc_pre) {
        ensure_dynamic_smem(k_dc_start, DC_SMEM);
        k_dc_start<<<dim3((unsigned)((B->n_env + DC_ENVS - 1) / DC_ENVS), (unsigned)((G->d.n + 63) / 64)), 256, DC_SMEM, (cudaStream_t)stream>>>(G->d, *B);
        ++g_launches;
    }
    if (use_tree(G, B)) {
        OpfgGrid* Gm = const_cast<OpfgGrid*>(G);
        const bool dyn = G->d.n_dyn > 0 && B->yval;
        constexpr int T = TREE_LANES;
        // at most 24 environments take the register cap of 384 threads (155 instead of 128 registers).  Measured on
        // B200 (122-bus grid, 32 768 environments, the 18-level minimum-degree order): 0.80 instead of 0.90 ms --
        // under the 128-register cap the staged-table base addresses were recomputed at their use sites.  The
        // 14-level centre-rooted order changes neither the registers nor the environments per SM
        void (*fns[4])(GridDev, OpfgBatch, int, int) = {k_pf_tree<T, false, 512>, k_pf_tree<T, true, 512>,
                                                        k_pf_tree<T, false, 384>, k_pf_tree<T, true, 384>};
        if (!Gm->tree_attr_set) {      // per grid, hence per device
            for (auto* f : fns) cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
            Gm->tree_attr_set = true;
        }
        const int E = G->tree_E;
        const int64_t groups = (B->n_env + E - 1) / E;
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>(groups, G->n_sm));
        auto* fn = fns[(E <= 24 ? 2 : 0) + (dyn ? 1 : 0)];
        fn<<<grid, T * E, G->tree_smem, (cudaStream_t)stream>>>(tree_view(G->d), *B, E, (int)G->tree_env_doubles);
        ++g_launches;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail("pf_solve (radial) launch: %s", cudaGetErrorString(e));
        return 0;
    }
    if (use_lanes(G, B)) {
        OpfgGrid* Gm = const_cast<OpfgGrid*>(G);
        void (*fns[8])(GridDev, OpfgBatch, double*, size_t) = {
            k_pf_lanes<0>, k_pf_lanes<1>, k_pf_lanes<2>, k_pf_lanes<3>, k_pf_lanes<4>, k_pf_lanes<5>, k_pf_lanes<6>, k_pf_lanes<7>};
        if (!Gm->lane_attr_set) {      // per grid, hence per device (function attributes are per device)
            for (auto* f : fns) cudaFuncSetAttribute(f, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
            Gm->lane_attr_set = true;
        }
        const GridDev view = lane_view(G->d, G->lane_stage != 0);
        const int64_t groups = (B->n_env + 31) / 32;
        // as many CTAs as there is work for W warps each, at most one per SM
        const int W = G->lane_warps_per_cta;
        const unsigned grid = (unsigned)std::max<int64_t>(1, std::min<int64_t>((groups + W - 1) / W, G->lane_ctas));
        auto* fn = fns[(G->lane_stage ? 1 : 0) | (G->d.n_qlim > 0 ? 2 : 0) | ((G->d.n_dyn > 0 && B->yval) ? 4 : 0)];
        fn<<<grid, 32 * W, G->lane_smem, (cudaStream_t)stream>>>(view, *B, G->lane_scratch, G->lane_warp_doubles);
        ++g_launches;
        cudaError_t e = cudaGetLastError();
        if (e != cudaSuccess) return fail("pf_solve (lanes) launch: %s", cudaGetErrorString(e));
        return 0;
    }
    const size_t smem = G->smem_pf;
    OPFG_DISPATCH_T(G->d.threads, {
        ensure_dynamic_smem(k_pf<TT>, smem);
        if (G->envs_per_cta > 1) {
            const int E = G->envs_per_cta;
            const size_t smem_multi = G->d.tab_staged_bytes + (size_t)E * smem;
            const int n_sm = current_sm_count();
            const int64_t groups = (B->n_env + E - 1) / E;
            const unsigned grid = (unsigned)std::min<int64_t>(groups, n_sm);
            const int stage = G->stage_level;
            const GridDev view = staged_view(G->d, stage);
            const int env_doubles = (int)(smem / 8);
            void (*fn)(GridDev, OpfgBatch, int, int) = nullptr;
            const int bound = TT * E <= 256 ? 256 : (TT * E <= 384 ? 384 : 768);   // 384 = three HV environments of 128 threads: 168 registers
            switch (stage | ((G->d.n_dyn > 0 && B->yval) ? 4 : 0)) {
                case 0: fn = pick_multi<TT, 0>(bound); break;
                case 1: fn = pick_multi<TT, 1>(bound); break;
                case 2: fn = pick_multi<TT, 2>(bound); break;
                case 4: fn = pick_multi<TT, 4>(bound); break;
                case 5: fn = pick_multi<TT, 5>(bound); break;
                default: fn = pick_multi<TT, 6>(bound); break;
            }
            ensure_dynamic_smem(fn, smem_multi);
            fn<<<grid, TT * E, smem_multi, (cudaStream_t)stream>>>(view, *B, E, env_doubles);
        } else {
            k_pf<TT><<<(unsigned)B->n_env, TT, smem, (cudaStream_t)stream>>>(G->d, *B);
        }
    });
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("pf_solve launch: %s", cudaGetErrorString(e));
#endif
    return 0;
}

int opfg_score(const OpfgGrid* G, const OpfgBatch* B, void* stream) {
    if (!G || !B) return fail("null argument");
    if (!G->has_scoring) return fail("opfg_set_scoring was not called");
    if (!B->state || !B->sbus || !B->vm || !B->va || !B->converged) return fail("opfg_score needs state, sbus, vm, va, converged");
    if (B->n_env <= 0) return 0;
#ifdef OPFG_HOSTSIM
    (void)stream;
    Ctx<1> cx;
    std::vector<double> sm(score_smem_doubles(G->d.nb, G->d.nbr, 32));
    for (int64_t env = 0; env < B->n_env; ++env)
        env_score(G->d, cx, sm.data(), *B, env,
                  (G->d.n_dyn > 0 && B->yval) ? B->yval + env * (int64_t)G->d.nnz_y * 2 : nullptr,
                  B->state + env * (int64_t)G->d.n_state);
#else
    const size_t smem = score_smem_doubles(G->d.nb, G->d.nbr, G->score_threads) * sizeof(double);
    if (G->score_threads == 32) {
        const size_t per_env = (smem + 15) & ~size_t(15);
        ensure_dynamic_smem(k_score_warps, per_env * 2);
        k_score_warps<<<(unsigned)((B->n_env + 1) / 2), 64, per_env * 2, (cudaStream_t)stream>>>(G->d, *B, (int)(per_env / 8));
    } else {
        const int T = G->score_threads;
        void (*fn)(GridDev, OpfgBatch) = T == 64 ? k_score<64> : (T == 128 ? k_score<128> : (T == 256 ? k_score<256> : nullptr));
        if (!fn) return fail("unsupported threads_per_env %d", T);
        ensure_dynamic_smem(fn, smem);
        fn<<<(unsigned)B->n_env, T, smem, (cudaStream_t)stream>>>(G->d, *B);
    }
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("score launch: %s", cudaGetErrorString(e));
#endif
    return 0;
}

// ---- mixed batch: kernel 1 / kernel 5 of several grids in one launch each ----
struct OpfgMixed {
    int n = 0;
    std::vector<const OpfgGrid*> grids;
    std::vector<MixedMember> host;
    void* dev = nullptr;
    int ctas_assemble = 0, ctas_score = 0;
    size_t smem_score = 0;
    ~OpfgMixed() { dev_free(dev); }
};

int opfg_mixed_create(int32_t n_members, const OpfgGrid* const* grids, const OpfgBatch* batches, OpfgMixed** out) {
    if (!out || !grids || !batches || n_members <= 0 || n_members > OPFG_MAX_MEMBERS) return fail("bad argument (1..8 members)");
    *out = nullptr;
    auto M = std::make_unique<OpfgMixed>();
    M->n = n_members;
    for (int m = 0; m < n_members; ++m) {
        const OpfgGrid* G = grids[m];
        if (!G || !G->has_assembly || !G->has_scoring) return fail("member %d: opfg_set_assembly / opfg_set_scoring missing", m);
        const OpfgBatch& B = batches[m];
        if (!B.state || !B.sbus || !B.vm || !B.va || !B.converged) return fail("member %d: batch needs state, sbus, vm, va, converged", m);
        if (G->d.n_dyn > 0 && (!B.yval || !B.bry)) return fail("member %d: grid has dynamic branches: batch needs yval and bry", m);
        M->grids.push_back(G);
        MixedMember mm{};
        mm.g = G->d; mm.B = B;
        mm.score_threads = G->score_threads == 32 ? 32 : 128;
        if (G->score_threads != 32 && G->score_threads != 128) return fail("member %d: scoring with %d threads per environment cannot join a mixed launch", m, G->score_threads);
        const size_t per_env = (score_smem_doubles(G->d.nb, G->d.nbr, mm.score_threads) * sizeof(double) + 15) & ~size_t(15);
        mm.score_env_doubles = (int)(per_env / 8);
        M->smem_score = std::max(M->smem_score, mm.score_threads == 32 ? 4 * per_env : per_env);
        M->host.push_back(mm);
    }
    M->dev = dev_alloc(sizeof(MixedMember) * n_members);
    if (!M->dev) return fail("device allocation failed");
    *out = M.release();
    return 0;
}

void opfg_mixed_destroy(OpfgMixed* mixed) { delete mixed; }

// which = 0: kernel 1 (opfg_assemble of every member), 1: kernel 5 (opfg_score of every member); the
// batches are re-read at every call (state double-buffering moves the pointers)
static int mixed_launch(OpfgMixed* M, const OpfgBatch* batches, int which, void* stream) {
    if (!M || !batches) return fail("null argument");
    int cta = 0;
    for (int m = 0; m < M->n; ++m) {
        MixedMember& mm = M->host[m];
        mm.B = batches[m];
        const int per_cta = (which == 0 || mm.score_threads == 32) ? 4 : 1;
        mm.cta_begin = cta;
        cta += (int)((mm.B.n_env + per_cta - 1) / per_cta);
        mm.cta_end = cta;
    }
    if (cta == 0) return 0;
#ifdef OPFG_HOSTSIM
    (void)stream;
    for (int m = 0; m < M->n; ++m) {
        const int rc = which == 0 ? opfg_assemble(M->grids[m], &M->host[m].B, nullptr) : opfg_score(M->grids[m], &M->host[m].B, nullptr);
        if (rc) return rc;
    }
#else
    // the member table travels on the same stream as the launch (a few KB)
    cudaMemcpyAsync(M->dev, M->host.data(), sizeof(MixedMember) * M->n, cudaMemcpyHostToDevice, (cudaStream_t)stream);
    if (which == 0) {
        k_assemble_mixed<<<cta, 128, 0, (cudaStream_t)stream>>>((const MixedMember*)M->dev, M->n);
    } else {
        ensure_dynamic_smem(k_score_mixed, M->smem_score);
        k_score_mixed<<<cta, 128, M->smem_score, (cudaStream_t)stream>>>((const MixedMember*)M->dev, M->n);
    }
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("mixed launch: %s", cudaGetErrorString(e));
#endif
    return 0;
}

int opfg_assemble_mixed(OpfgMixed* mixed, const OpfgBatch* batches, void* stream) { return mixed_launch(mixed, batches, 0, stream); }
int opfg_score_mixed(OpfgMixed* mixed, const OpfgBatch* batches, void* stream) { return mixed_launch(mixed, batches, 1, stream); }

int opfg_observe(const OpfgGrid* G, const OpfgBatch* B, void* stream) {
    if (!G || !B) return fail("null argument");
    if (!G->has_scoring) return fail("opfg_set_scoring was not called");
    if (!B->state || (!B->obs_f32 && !B->obs_f64)) return fail("opfg_observe needs state and an obs buffer");
    if (B->n_env <= 0 || G->d.n_obs == 0) return 0;
#ifdef OPFG_HOSTSIM
    (void)stream;
    for (int64_t env = 0; env < B->n_env; ++env)
        for (int j = 0; j < G->d.n_obs; ++j) {
            const double v = obs_value(G->d, B->state + env * (int64_t)G->d.n_state, j);
            if (B->obs_f32) B->obs_f32[env * G->d.n_obs + j] = (float)v;
            if (B->obs_f64) B->obs_f64[env * G->d.n_obs + j] = v;
        }
#else
    const ItemGrid ig = item_grid(B->n_env, G->d.n_obs);
    k_observe<<<ig.grid, 256, 0, (cudaStream_t)stream>>>(G->d, *B, ig.w_log2);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("observe launch: %s", cudaGetErrorString(e));
#endif
    return 0;
}

#ifdef OPFG_PHASE_TIMING
/* developer instrumentation: cycles of thread 0 per phase, summed over CTAs (8 slots) */
extern "C" int opfg_debug_phase_cycles(OpfgGrid* G, unsigned long long* host_out, int reset) {
    if (!G->d.phase_cycles) G->d.phase_cycles = (unsigned long long*)G->up(std::vector<unsigned long long>(144, 0ull));
    cudaDeviceSynchronize();
    if (host_out) cudaMemcpy(host_out, G->d.phase_cycles, 144 * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
    if (reset) cudaMemset(G->d.phase_cycles, 0, 144 * sizeof(unsigned long long));
    return 0;
}
#endif

int opfg_row_program_create(int32_t n_rows, int32_t n_ops, const OpfgRowOp* ops, int32_t n_static,
                            const double* statics, OpfgRowProgram** out) {
    if (!ops || !out || n_rows < 0 || n_ops <= 0 || n_ops > 96) return fail("bad row program (1..96 ops)");
    for (int i = 0; i < n_ops; ++i) {
        const OpfgRowOp& o = ops[i];
        const bool reg_ok = o.dst >= 0 && o.dst < 16;
        if (o.op < 0 || o.op > OPFG_OP_STORE_STATE) return fail("row program: unknown op %d", o.op);
        if (o.op != OPFG_OP_STORE_STATE && !reg_ok) return fail("row program: register out of range");
        if (o.op >= OPFG_OP_ADD && o.op != OPFG_OP_STORE_STATE && (o.a < 0 || o.a >= 16)) return fail("row program: bad operand");
        if (o.op == OPFG_OP_STORE_STATE && (o.b < 0 || o.b >= 16)) return fail("row program: bad store register");
        if (o.op == OPFG_OP_LOAD_STATIC && (o.a < 0 || o.a + n_rows > n_static)) return fail("row program: static out of range");
        if ((o.op == OPFG_OP_LOAD_STATE || o.op == OPFG_OP_STORE_STATE) && o.a < 0) return fail("row program: negative state cell");
    }
    auto* P = new OpfgRowProgram();
    P->n_rows = n_rows; P->n_ops = n_ops; P->n_items = n_rows;
    for (int i = 0; i < n_ops; ++i) {
        if (ops[i].op != OPFG_OP_STORE_STATE) P->n_regs = std::max(P->n_regs, ops[i].dst + 1);
        if (ops[i].op == OPFG_OP_LOAD_STATE || ops[i].op == OPFG_OP_STORE_STATE) P->max_a = std::max(P->max_a, ops[i].a);
    }
    P->max_cell = P->max_a >= 0 && n_rows > 0 ? P->max_a + n_rows - 1 : -1;
    P->host_ops.assign(ops, ops + n_ops);
    P->host_statics.assign(statics, statics + n_static);
    P->ops = (OpfgRowOp*)dev_alloc(sizeof(OpfgRowOp) * n_ops);
    P->statics = (double*)dev_alloc(sizeof(double) * std::max(n_static, 1));
    dev_put(P->ops, ops, sizeof(OpfgRowOp) * n_ops);
    dev_put(P->statics, statics, sizeof(double) * n_static);
    *out = P;
    return 0;
}

void opfg_row_program_destroy(OpfgRowProgram* p) { delete p; }

int opfg_row_program_select_rows(OpfgRowProgram* P, int32_t n_sel, const int32_t* rows) {
    if (!P || n_sel < 0 || (n_sel > 0 && !rows)) return fail("bad argument");
    for (int i = 0; i < n_sel; ++i)
        if (rows[i] < 0 || rows[i] >= P->n_rows) return fail("row program: selected row %d out of range", rows[i]);
    dev_free(P->rows);
    P->rows = (int32_t*)dev_alloc(sizeof(int32_t) * std::max(n_sel, 1));
    if (!P->rows) return fail("device allocation failed");
    dev_put(P->rows, rows, sizeof(int32_t) * n_sel);
    P->host_rows.assign(rows, rows + n_sel);
    P->n_items = n_sel;
    const int max_row = n_sel > 0 ? *std::max_element(rows, rows + n_sel) : -1;
    P->max_cell = P->max_a >= 0 && max_row >= 0 ? P->max_a + max_row : -1;
    return 0;
}

int opfg_row_program_run(const OpfgRowProgram* P, int64_t n_env, double* state, int32_t n_state, void* stream) {
    if (!P || !state || n_env < 0) return fail("bad argument");
    if (P->max_cell >= n_state) return fail("row program touches cell %d of a %d-cell state row", P->max_cell, n_state);
    if (n_env == 0 || P->n_items == 0) return 0;
#ifdef OPFG_HOSTSIM
    (void)stream;
    for (int64_t env = 0; env < n_env; ++env)
        for (int item = 0; item < P->n_items; ++item)
            { double r[16]; row_program_exec(P->ops, P->n_ops, P->statics, P->rows ? P->rows[item] : item, state + env * (int64_t)n_state, r, 1); }
#else
    const ItemGrid ig = item_grid(n_env, P->n_items);
    k_row_program<<<ig.grid, 256, sizeof(double) * 256 * P->n_regs, (cudaStream_t)stream>>>(
        P->ops, P->n_ops, P->statics, P->n_items, P->rows, n_env, state, n_state, ig.w_log2);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("row program launch: %s", cudaGetErrorString(e));
#endif
    return 0;
}

int opfg_reset_plan_create(const OpfgResetStage* stages, int32_t n_stages, OpfgResetPlan** out) {
    if (!out || n_stages < 0 || (n_stages > 0 && !stages)) return fail("bad argument");
    *out = nullptr;
    static_assert(sizeof(ResetStage) % 8 == 0 && sizeof(OpfgRowOp) == 24, "staging copies whole doubles");
    try {
        auto P = std::make_unique<OpfgResetPlan>();
        for (int k = 0; k < n_stages; ++k) {
            const OpfgResetStage& a = stages[k];
            ResetStage s{};
            std::vector<int> rd, wr;
            s.kind = a.kind;
            if (a.kind == 0) {
                if (!a.slots || !a.lo || !a.hi || !a.div || a.n_cols < 0) return fail("reset stage %d: bad sampler arrays", k);
                s.n_cols = a.n_cols; s.slots = a.slots; s.lo = a.lo; s.hi = a.hi; s.dv = a.div;
                s.stream_off = a.stream_offset;
                wr.resize(a.n_cols);
#ifdef OPFG_HOSTSIM
                memcpy(wr.data(), a.slots, sizeof(int) * a.n_cols);
#else
                cudaMemcpy(wr.data(), a.slots, sizeof(int) * a.n_cols, cudaMemcpyDeviceToHost);
#endif
            } else if (a.kind == 1) {
                if (!a.program) return fail("reset stage %d: null row program", k);
                const OpfgRowProgram& rp = *a.program;
                s.ops = rp.ops; s.statics = rp.statics;   // device copies (host memory in the host build)
                s.n_ops = rp.n_ops; s.n_rows = rp.n_items; s.rows = rp.rows;
                s.ops_smem = P->n_ops_total;
                P->n_ops_total += rp.n_ops;
                P->n_regs = std::max(P->n_regs, rp.n_regs);
                for (const OpfgRowOp& o : rp.host_ops)
                    if (o.op == OPFG_OP_LOAD_STATE || o.op == OPFG_OP_STORE_STATE)
                        for (int it = 0; it < rp.n_items; ++it)
                            (o.op == OPFG_OP_LOAD_STATE ? rd : wr).push_back(o.a + (rp.host_rows.empty() ? it : rp.host_rows[it]));
            } else return fail("reset stage %d: unknown kind %d", k, a.kind);
            for (int c : wr) { if (c < 0) return fail("reset stage %d: negative state cell", k); P->max_cell = std::max(P->max_cell, c); }
            for (int c : rd) { if (c < 0) return fail("reset stage %d: negative state cell", k); P->max_cell = std::max(P->max_cell, c); }
            std::sort(rd.begin(), rd.end()); std::sort(wr.begin(), wr.end());
            P->host.push_back(s); P->reads.push_back(rd); P->writes.push_back(wr);
        }
        // stages that touch disjoint cells run side by side (no barrier, items spread over the threads)
        auto overlap = [](const std::vector<int>& a, const std::vector<int>& b) {
            size_t i = 0, j = 0;
            while (i < a.size() && j < b.size()) { if (a[i] == b[j]) return true; if (a[i] < b[j]) ++i; else ++j; }
            return false;
        };
        int group_begin = 0, items = 0;
        for (int k = 0; k < n_stages; ++k) {
            ResetStage& s = P->host[k];
            bool independent = true;
            for (int j = group_begin; j < k && independent; ++j)
                independent = !overlap(P->writes[j], P->reads[k]) && !overlap(P->writes[j], P->writes[k]) &&
                              !overlap(P->reads[j], P->writes[k]);
            if (!independent) { P->host[k - 1].sync_after = 1; group_begin = k; items = 0; }
            s.item_off = items;
            items += s.kind == 0 ? (s.n_cols + 1) / 2 : s.n_rows;
        }
        if (n_stages > 0) P->host[n_stages - 1].sync_after = 1;
        P->dev = (ResetStage*)dev_alloc(sizeof(ResetStage) * P->host.size());
        if (!P->dev) return fail("device allocation failed");
        dev_put(P->dev, P->host.data(), sizeof(ResetStage) * P->host.size());
        *out = P.release();
    } catch (const std::exception& e) { return fail("opfg_reset_plan_create: %s", e.what()); }
    return 0;
}

void opfg_reset_plan_destroy(OpfgResetPlan* plan) { delete plan; }

int opfg_reset_episode(const OpfgGrid* G, const OpfgBatch* B, const OpfgResetPlan* P_, uint64_t seed, uint64_t first_env,
                       uint64_t stream_base, int32_t random_action, uint32_t action_stream_offset, void* stream) {
    if (!G || !B || !P_) return fail("null argument");
    OpfgResetPlan* P = const_cast<OpfgResetPlan*>(P_);
    if (!G->has_assembly || !G->has_scoring) return fail("opfg_reset_episode needs opfg_set_assembly and opfg_set_scoring");
    if (!B->state || !B->actions || (!B->obs_f32 && !B->obs_f64)) return fail("opfg_reset_episode needs state, actions and an obs buffer");
    if (P->max_cell >= G->d.n_state) return fail("reset plan touches cell %d of a %d-cell state row", P->max_cell, G->d.n_state);
    if (B->n_env <= 0) return 0;
    const int n_st = (int)P->host.size();
#ifdef OPFG_HOSTSIM
    (void)stream;
    Ctx<1> cx;
    double host_regs[16];
    for (int64_t env = 0; env < B->n_env; ++env)
        env_reset(G->d, cx, *B, env, B->state + env * (int64_t)G->d.n_state, P->host.data(), n_st, (const OpfgRowOp*)nullptr,
                  host_regs, 1, seed, first_env, stream_base, random_action, action_stream_offset);
#else
    const int n_in = G->d.n_inputs;
    if (P->for_inputs != n_in) {
        // The row needs no copy-in if every input cell is written before anything reads it: the first stage that
        // touches a cell must write it and not read it (a stage that does both may read first, as in a += 1)
        enum : char { UNTOUCHED, WRITTEN_FIRST, READ_FIRST };
        std::vector<char> first(std::max(n_in, 1), UNTOUCHED);
        for (size_t k = 0; k < P->host.size(); ++k) {
            for (int c : P->reads[k]) if (c < n_in && first[c] == UNTOUCHED) first[c] = READ_FIRST;
            for (int c : P->writes[k]) if (c < n_in && first[c] == UNTOUCHED) first[c] = WRITTEN_FIRST;
        }
        bool all = true;
        for (int c = 0; c < n_in && all; ++c) all = first[c] == WRITTEN_FIRST;
        P->covers_all = all; P->for_inputs = n_in;
    }
    // the row lives in shared memory if everything the reset touches lies in the input part
    const bool staged = n_in > 0 && P->max_cell < n_in && G->act_ref_max < n_in && G->obs_ref_max < n_in;
    const int n_row = staged ? n_in : 0;
    constexpr int T = 128;
    const size_t smem = sizeof(double) * n_row + sizeof(ResetStage) * n_st + sizeof(OpfgRowOp) * P->n_ops_total +
                        sizeof(double) * T * P->n_regs;
    if (smem > 227 * 1024) return fail("reset: %zu bytes of shared memory per environment", smem);
    ensure_dynamic_smem(k_reset<T>, smem);
    k_reset<T><<<(unsigned)B->n_env, T, smem, (cudaStream_t)stream>>>(
        G->d, *B, P->dev, n_st, n_row, staged && !P->covers_all, P->n_ops_total, seed, first_env, stream_base,
        random_action, action_stream_offset);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("reset launch: %s", cudaGetErrorString(e));
#endif
    return 0;
}

int opfg_fp64_probe(int32_t n_blocks, int32_t iters, double* out, void* stream) {
    if (!out || n_blocks <= 0 || iters <= 0) return fail("bad argument");
#ifdef OPFG_HOSTSIM
    (void)stream;
    return fail("opfg_fp64_probe measures the GPU; not available in the host build");
#else
    k_fp64_probe<<<n_blocks, 256, 0, (cudaStream_t)stream>>>(iters, out);
    ++g_launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return fail("fp64 probe launch: %s", cudaGetErrorString(e));
    return 0;
#endif
}

int opfg_step(const OpfgGrid* G, const OpfgBatch* B, void* stream) {
    int rc = opfg_assemble(G, B, stream);
    if (rc) return rc;
    rc = opfg_pf_solve(G, B, stream);
    if (rc) return rc;
    return opfg_score(G, B, stream);
}

}  // extern "C"
