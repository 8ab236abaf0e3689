"""``from_pandapower(net)``: build the engine's grid tables from a REAL pandapower net by reading
the ppc that pandapower itself produced (``net._ppc`` after ``pp.runpp`` / ``pp.pd2ppc``), instead
of re-deriving it with ``opfgym_b200.ppc.PpcBuilder`` (which restates that conversion for the
in-repo ``Net`` container).  This is the last hop of INTEGRATION.md §1: with it the engine solves
exactly the matrices pandapower's own Newton-Raphson would solve (reference call site
``opfgym/opf_env.py:703``).

STATUS: pandapower is not installable in the build image: against the real package this module is exercised only
by ``tests/parity/test_vs_pandapower.py``, which skips without pandapower; ``tests/test_pandapower_adapter_stub.py``
runs it against a ``net._ppc`` / ``net._pd2ppc_lookups`` laid out the way the notes below describe (built from the
oracle's own conversion), so that at least the reading logic is executed here.  Everything taken from
pandapower's private attributes is marked [ext-mem] (from memory of pandapower 2.13/2.14):

* ``net._ppc``: the external-numbered ppc -- ``bus``, ``gen``, ``branch`` (PYPOWER column order), ``baseMVA``;
  out-of-service / isolated buses carry ``BUS_TYPE == 4``, dead branches ``BR_STATUS == 0``.
* ``net._pd2ppc_lookups["bus"]``: array, pandapower bus index -> ppc bus row (fused buses share one).
* ``net._pd2ppc_lookups["branch"]``: dict, element table -> (first, last+1) row range in ``ppc["branch"]``.
* gen rows: ext_grids in table order first, then gens (``build_gen.py``); cross-checked through the bus.
* the shunt branch admittance: complex ``BR_B`` (``y = 1j * BR_B``) in pandapower < 2.14, a separate real
  ``BR_G`` column afterwards.
* ``net._pd2ppc_lookups["branch"]["trafo3w"]``: 3 rows per element, in blocks -- every element's hv->star row,
  then every mv row (star->mv), then every lv row (star->lv) (``build_branch._trafo_df_from_trafo3w``).  Loading
  of element k is the largest of the three outer-end currents (hv: the row's from bus, mv / lv: its to bus), each
  scaled by ``vn_<side>_kv / sn_<side>_mva`` (``results_branch._get_trafo3w_results``).
"""
from __future__ import annotations

import numpy as np

from . import ppc as P


class PandapowerPpcBuilder:
    """Same interface as ``opfgym_b200.ppc.PpcBuilder`` (``build``, ``element_bus``), fed by pandapower."""

    def __init__(self, net, **runpp_kwargs):
        if getattr(net, "_ppc", None) is None or net._ppc.get("bus") is None:
            import pandapower as pp                   # fails loudly where pandapower is absent
            kw = dict(enforce_q_lims=True)
            kw.update(runpp_kwargs)
            try:
                pp.runpp(net, **kw)                   # fills net._ppc / net._pd2ppc_lookups
            except pp.powerflow.LoadflowNotConverged:
                pass                                  # the tables exist even if this operating point diverges
        self._read(net)

    def _read(self, net):
        ppc = net._ppc
        bus_x, gen_x, br_x = np.asarray(ppc["bus"]), np.asarray(ppc["gen"]), np.asarray(ppc["branch"])
        keep_bus = bus_x[:, P.BUS_TYPE].real != P.NONE
        new_of = -np.ones(len(bus_x), dtype=np.int64)
        new_of[keep_bus] = np.arange(int(keep_bus.sum()))
        lookup = np.asarray(net._pd2ppc_lookups["bus"])
        pp_index = net.bus.index.to_numpy()
        self.bus_lookup = np.array([new_of[lookup[i]] if 0 <= i < len(lookup) and lookup[i] >= 0 else -1
                                    for i in pp_index], dtype=np.int64)
        self._pos_of = {int(b): k for k, b in enumerate(pp_index)}
        self.nb = int(keep_bus.sum())
        bus = np.zeros((self.nb, P.BUS_COLS))
        ncol = min(P.BUS_COLS, bus_x.shape[1])
        bus[:, :ncol] = bus_x[keep_bus][:, :ncol].real
        bus[:, P.BUS_I] = np.arange(self.nb)

        f = new_of[br_x[:, P.F_BUS].real.astype(int)]
        t = new_of[br_x[:, P.T_BUS].real.astype(int)]
        keep_br = (br_x[:, P.BR_STATUS].real != 0) & (f >= 0) & (t >= 0)
        row_of = -np.ones(len(br_x), dtype=np.int64)
        row_of[keep_br] = np.arange(int(keep_br.sum()))
        branch = np.zeros((int(keep_br.sum()), P.BRANCH_COLS))
        src = br_x[keep_br]
        for col in (P.BR_R, P.BR_X, P.RATE_A, P.TAP, P.SHIFT, P.BR_STATUS, P.ANGMIN, P.ANGMAX):
            branch[:, col] = src[:, col].real
        branch[:, P.F_BUS], branch[:, P.T_BUS] = f[keep_br], t[keep_br]
        if np.iscomplexobj(br_x):                      # y_shunt = 1j * BR_B  [ext-mem]
            y = 1j * src[:, P.BR_B]
            branch[:, P.BR_G], branch[:, P.BR_B] = y.real, y.imag
        else:
            branch[:, P.BR_B] = src[:, P.BR_B]
            # pandapower >= 2.14 keeps the conductance in a column of its own, whose index only pandapower knows:
            # no silent guess (a dropped conductance would be a different network)
            from pandapower.pypower.idx_brch import BR_G as PP_BR_G
            branch[:, P.BR_G] = src[:, PP_BR_G].real

        ranges = net._pd2ppc_lookups.get("branch", {})
        def element_rows(table):
            out = -np.ones(len(net[table]), dtype=np.int64)
            if table in ranges and len(net[table]):
                a, b = ranges[table]
                out[:] = row_of[a:b]
            return out
        self.line_branch, self.trafo_branch = element_rows("line"), element_rows("trafo")

        g_bus = new_of[gen_x[:, P.GEN_BUS].real.astype(int)]
        keep_gen = (gen_x[:, P.GEN_STATUS].real > 0) & (g_bus >= 0)
        gen = np.zeros((int(keep_gen.sum()), P.GEN_COLS))
        ncol = min(P.GEN_COLS, gen_x.shape[1])
        gen[:, :ncol] = gen_x[keep_gen][:, :ncol].real
        gen[:, P.GEN_BUS] = g_bus[keep_gen]
        gen_row = -np.ones(len(gen_x), dtype=np.int64)
        gen_row[keep_gen] = np.arange(int(keep_gen.sum()))
        n_eg = len(net.ext_grid)
        self.ext_grid_gen = gen_row[:n_eg].copy()
        self.gen_gen = gen_row[n_eg:n_eg + len(net.gen)].copy() if len(net.gen) else np.zeros(0, np.int64)
        for table, rows in (("ext_grid", self.ext_grid_gen), ("gen", self.gen_gen)):
            want = self.element_bus(net, table)
            for k, r in enumerate(rows):
                if r >= 0 and int(gen[r, P.GEN_BUS]) != want[k]:
                    raise RuntimeError(f"{table} row order in net._ppc['gen'] is not the assumed one [ext-mem]")

        # loading factors (results_branch.py [ext-mem]): same formulas as PpcBuilder.branch_table
        rate_f, rate_t = np.zeros(len(branch)), np.zeros(len(branch))
        base_kv = bus[:, P.BASE_KV]
        for pos, r in enumerate(self.line_branch):
            if r >= 0:
                ln = net.line.iloc[pos]
                imax = float(ln.max_i_ka) * float(ln.df) * float(ln.parallel)
                rate_f[r] = 1.0 / (np.sqrt(3.0) * base_kv[int(branch[r, P.F_BUS])] * imax)
                rate_t[r] = 1.0 / (np.sqrt(3.0) * base_kv[int(branch[r, P.T_BUS])] * imax)
        for pos, r in enumerate(self.trafo_branch):
            if r >= 0:
                tr = net.trafo.iloc[pos]
                cap = float(tr.sn_mva) * float(tr.parallel) * float(tr.df)
                rate_f[r] = float(tr.vn_hv_kv) / (base_kv[int(branch[r, P.F_BUS])] * cap)
                rate_t[r] = float(tr.vn_lv_kv) / (base_kv[int(branch[r, P.T_BUS])] * cap)
        # trafo3w: three rows per element behind its star-point bus, loading factors at the outer ends only
        n3 = len(net.trafo3w) if "trafo3w" in net else 0
        self.trafo3w_branch = -np.ones((n3, 3), dtype=np.int64)
        if n3 and "trafo3w" in ranges:
            a, b = ranges["trafo3w"]
            if b - a != 3 * n3:
                raise RuntimeError("net._ppc['branch'] does not hold 3 rows per trafo3w [ext-mem]")
            self.trafo3w_branch[:] = row_of[a:b].reshape(3, n3).T
            for pos, rows in enumerate(self.trafo3w_branch):
                t3 = net.trafo3w.iloc[pos]
                for w, (side, end) in enumerate((("hv", P.F_BUS), ("mv", P.T_BUS), ("lv", P.T_BUS))):
                    r = rows[w]
                    if r < 0:
                        continue
                    rate = float(t3[f"vn_{side}_kv"]) / (base_kv[int(branch[r, end])] * float(t3[f"sn_{side}_mva"]))
                    (rate_f if end == P.F_BUS else rate_t)[r] = rate
        # Branches of other element tables (impedance) are solved like any other row of pandapower's ppc; they have
        # no result rows here (no res_impedance cells, loading factors 0).  An xward also injects power at its bus,
        # which kernel 1 would not scatter: rejected.
        self.other_branch_rows = {}
        covered = (self.line_branch >= 0).sum() + (self.trafo_branch >= 0).sum() + (self.trafo3w_branch >= 0).sum()
        for table in ranges:
            if table in ("line", "trafo", "trafo3w"):
                continue
            a, b = ranges[table]
            rows = row_of[a:b][row_of[a:b] >= 0]
            if table == "xward" and b > a:
                raise NotImplementedError("net.xward: its constant-power part is not an injection kernel 1 knows")
            self.other_branch_rows[table] = rows
            covered += len(rows)
        if covered != keep_br.sum():
            raise NotImplementedError(f"{int(keep_br.sum() - covered)} rows of net._ppc['branch'] belong to no element "
                                      "table of net._pd2ppc_lookups['branch']")
        eg, gn = net.ext_grid, net.gen
        vm = np.concatenate([eg.vm_pu.to_numpy(float), gn.vm_pu.to_numpy(float) if len(gn) else np.zeros(0)])
        self._ppc = P.Ppc(base_mva=float(ppc["baseMVA"]), bus=bus, gen=gen, branch=branch,
                          bus_lookup=self.bus_lookup.copy(), line_branch=self.line_branch.copy(),
                          trafo_branch=self.trafo_branch.copy(), ext_grid_gen=self.ext_grid_gen,
                          gen_gen=self.gen_gen, rate_f=rate_f, rate_t=rate_t,
                          init_vm_pu=float(vm.mean()) if len(vm) else 1.0,
                          trafo3w_branch=self.trafo3w_branch.copy())

    def element_bus(self, net, table):
        pos = np.array([self._pos_of[int(b)] for b in net[table].bus.to_numpy()], dtype=np.int64)
        return self.bus_lookup[pos] if len(pos) else pos

    def build(self, net) -> P.Ppc:
        """Topology and branch parameters are pandapower's; the bus demand columns are irrelevant to the
        engine (kernel 1 scatters the injections from the element tables every step)."""
        return self._ppc


def from_pandapower(net, **runpp_kwargs) -> PandapowerPpcBuilder:
    return PandapowerPpcBuilder(net, **runpp_kwargs)
