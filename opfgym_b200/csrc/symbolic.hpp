// Host-side symbolic analysis, run once per grid (replaces the per-call
// COLAMD/AMD ordering that SuperLU/KLU perform inside pandapower's newtonpf /
// lightsim2grid, reference call site opfgym/opf_env.py:703  [ext-mem]).
//
// The Newton-Raphson Jacobian is handled as a matrix of 2x2 blocks, one block
// row/column per non-slack bus (unknowns (theta_i, |V|_i); PV buses keep an
// identity row for |V|).  Its block pattern equals the bus adjacency pattern,
// which is fixed for all environments, so ordering, fill and the parallel
// schedule are computed here once and shipped to the device as flat tables.
#pragma once
#include <cstdint>
#include <string>
#include <vector>

namespace opfg {

struct BranchHost {
    int f, t;              // ppc bus indices
    double r, x, b, g, tap, shift_deg;
};

struct Symbolic {
    int nb = 0;            // buses
    int n = 0;             // non-ref buses = pivots
    int n_levels = 0;
    std::vector<int> int_of_bus, bus_of_int;   // internal numbering: pivots in elimination order, then ref buses
    std::vector<int> level_ptr;                // [n_levels+1] pivot ranges per level
    // ---- blocks of the filled Jacobian: ids 0..n-1 are the diagonals (id == pivot) ----
    int n_blocks = 0;
    std::vector<int> blk_row, blk_col;
    std::vector<int> fill_ids;                 // blocks absent from the Ybus pattern (start at zero)
    // diag k: D_k -= L~(k,m) * W(m,k), y_k -= L~(k,m) * t_m   over pairs in increasing m
    std::vector<int> dp_ptr, dp_l, dp_w, dp_m;
    // eager gather: the pairs of pivot k whose source sits more than one level below k are applied
    // as soon as that source level is finished (phase = source level + 1), by an item of their own;
    // pivot k's own item starts at dp_own[k] (sources of the level right below) and inverts.
    std::vector<int> dp_own;                   // [n]
    std::vector<int> eg_ptr;                   // [n_levels+1] eager item ranges per diagonal phase
    std::vector<int> eg_k, eg_begin, eg_count; // target pivot, first pair, number of pairs
    // off-diagonal work items, grouped by level of their pivot
    std::vector<int> off_ptr;                  // [n_levels+1] item ranges
    std::vector<int> off_tgt, off_piv;         // target block; pivot whose inverse scales it (U blocks) or -1 (L blocks)
    std::vector<int> op_ptr, op_l, op_w;       // pairs per item
    // backward substitution: x_k = t_k - sum W(k,j) x_j
    std::vector<int> up_ptr, up_w, up_j;
    // ---- Ybus CSR in internal numbering (ref rows last) ----
    std::vector<int> y_ptr, y_col, y_blk;      // y_blk: Jacobian block fed by this entry (-1 if row/col is ref)
    std::vector<int> yc_ptr, yc_branch, yc_role;  // contributions: role 0..3 = ff, ft, tf, tt; 4 = bus shunt (branch = bus)
    std::vector<int> y_diag;                   // [nb] position of the diagonal entry of each row
    // ---- cost / flop model ----
    double lu_flops = 0, flops_per_iter = 0;
    double est_cycles = 0;
    std::string ordering_name;
};

// Row-wise (IKJ) form of the same factorisation, for the lane-per-environment kernel: row k of the
// filled Jacobian is built in a small row buffer -- L(k, m) for the earlier pivots m it touches,
// the diagonal, U(k, j) for the later ones --, the rows of the earlier pivots are eliminated from it
// in increasing m, and only W(k, j) = D_k^-1 U(k, j) and t_k leave the buffer.  Every sum runs in the
// order of the gather lists above, so both kernels produce the same bits.
struct LaneSchedule {
    int max_row = 0;                          // largest row pattern, in blocks
    std::vector<int> y_rpos;                  // per Ybus entry of the non-slack rows: row-buffer position, -1 = slack column
    std::vector<int> diag_pos;                // [n]
    std::vector<int> fill_ptr, fill_rpos;     // [n+1]; positions that start at zero (fill blocks)
    std::vector<int> el_ptr;                  // [n+1] elimination items of row k (ascending m)
    std::vector<int> el_rpos, el_m, el_uptr;  // position of L(k, m); m; its update range (el_uptr has one more entry)
    std::vector<int> upd_w, upd_rpos;         // W slot = position in the up_* lists; target position in the row buffer
    std::vector<int> up_rpos;                 // aligned with up_ptr / up_j: position of U(k, j)
};
void build_lane_schedule(const Symbolic& s, LaneSchedule& out);

// true when the graph of the non-reference buses (self loops and parallel branches dropped) is a forest:
// edges == nodes - components
bool is_forest(int nb, const std::vector<int>& bus_type, const std::vector<BranchHost>& branches);

// ordering: 0 auto (cheapest by the CTA kernel's cost model), 1 minimum degree, 2 independent-set rounds,
// 3 least work (fewest Schur-update pairs; what the lane-per-environment kernel wants), 4 leaf-first with
// every tree rooted at its centre (forests only: no fill, radius + 1 levels per tree; the radial kernel's order)
// level_cap > 0 (centre-rooted order only): at most that many pivots per level (balanced levels)
void analyse(int nb, const std::vector<int>& bus_type, const std::vector<BranchHost>& branches,
             int ordering, int threads_per_env, Symbolic& out, int level_cap = 0);

// scalar LU of the DC matrix B'[nonref, nonref] on the same schedule.
// Outputs indexed by block id: inv_d[k] (k<n), val[id] = W for U blocks, L~ for L blocks.
void factor_dc(const Symbolic& s, const std::vector<BranchHost>& branches,
               std::vector<double>& dc_val, bool& ok);

}  // namespace opfg
