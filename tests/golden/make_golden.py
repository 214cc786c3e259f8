"""Generates the committed golden fixtures from the reference tree (run once, here, where
/root/reference exists):

  pp_results_<env>.json   the res_* tables real pandapower stored in grid2op/data/<env>/grid.json
  case14_sandbox_chronics.npz   float32 load_p/load_q/prod_p/prod_v rows of the 3 bundled scenarios of
                          l2rpn_case14_sandbox re-ordered to BACKEND element order (bench / series tests)
  oracle_case14_steps.npz  oracle (fp64) results on 64 chronics rows of l2rpn_case14_sandbox
"""
import bz2
import json
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
from oracle import pandapower_ref as ppr  # noqa: E402
from grid2op_b200.gridmodel import GridModel  # noqa: E402

REF = os.environ.get("GRID2OP_REF_DATA", "/root/reference/grid2op/data")
COLS = {
    "bus": ["vm_pu", "va_degree"],
    "line": ["p_from_mw", "q_from_mvar", "p_to_mw", "q_to_mvar", "i_from_ka", "i_to_ka", "vm_from_pu", "va_from_degree",
             "vm_to_pu", "va_to_degree"],
    "trafo": ["p_hv_mw", "q_hv_mvar", "p_lv_mw", "q_lv_mvar", "i_hv_ka", "i_lv_ka"],
    "gen": ["p_mw", "q_mvar", "vm_pu", "va_degree"],
}


def stored_results():
    for env in ("rte_case5_example", "l2rpn_neurips_2020_track1", "l2rpn_wcci_2022_dev"):
        net = ppr.from_json(os.path.join(REF, env, "grid.json"))
        out = {"env": env, "res": {}}
        for tab, cols in COLS.items():
            st = net.stored_res.get("res_" + tab)
            if st is None or len(st) == 0:
                continue
            out["res"][tab] = {c: [None if not np.isfinite(v) else float(v) for v in st.num(c, np.nan)] for c in cols if c in st}
        with open(os.path.join(HERE, f"pp_results_{env}.json"), "w") as f:
            json.dump(out, f)


def read_csv_bz2(path):
    with bz2.open(path, "rt") as f:
        header = f.readline().strip().split(";")
        rows = [[float(x) for x in line.strip().split(";")] for line in f if line.strip()]
    return header, np.array(rows, dtype=np.float64)


def case14_chronics():
    env = "l2rpn_case14_sandbox"
    gm = GridModel(os.path.join(REF, env, "grid.json"))
    scen = []
    for sc in ("0000", "0001", "0002"):
        d = os.path.join(REF, env, "chronics", sc)
        cols = []
        for fn, names in (("load_p", gm.name_load), ("load_q", gm.name_load), ("prod_p", gm.name_gen), ("prod_v", gm.name_gen)):
            hdr, arr = read_csv_bz2(os.path.join(d, fn + ".csv.bz2"))
            order = [hdr.index(n) for n in names]            # chronics columns are matched by NAME
            cols.append(arr[:, order])
        scen.append(np.concatenate(cols, axis=1).astype(np.float32))
    chron = np.stack(scen)                                    # [3, 576, 2*n_load + 2*n_gen]
    np.savez_compressed(os.path.join(HERE, "case14_sandbox_chronics.npz"), chron=chron,
                        name_load=gm.name_load, name_gen=gm.name_gen)
    return gm, chron


def grid_models():
    for env in ("l2rpn_case14_sandbox", "rte_case5_example", "l2rpn_neurips_2020_track1", "l2rpn_wcci_2022_dev"):
        gm = GridModel(os.path.join(REF, env, "grid.json"))
        gm.path = env            # no absolute paths in fixtures
        gm.to_npz(os.path.join(HERE, f"gridmodel_{env}.npz"))


def oracle_steps(gm, chron, n=48):
    """fp64 oracle results for n (scenario,row) pairs of the case14 chronics: the parity fixture the GPU
    box checks the CUDA path against when the reference tree is absent."""
    sys.path.insert(0, os.path.join(os.path.dirname(HERE)))
    from oracle_engine import OracleEngine
    gm_full = GridModel(os.path.join(REF, "l2rpn_case14_sandbox", "grid.json"))
    eng = OracleEngine(gm_full)
    sl = gm_full.inj_slices()
    rng = np.random.default_rng(0)
    scen = rng.integers(0, chron.shape[0], n)
    rows = rng.integers(0, chron.shape[1], n)
    inj = np.tile(gm_full.default_inj(), (n, 1))
    nl, ng = gm_full.n_load, gm_full.n_gen
    for i in range(n):
        r = chron[scen[i], rows[i]]
        inj[i, sl["load_p"]] = r[:nl]
        inj[i, sl["load_q"]] = r[nl:2 * nl]
        inj[i, sl["gen_p"]] = r[2 * nl:2 * nl + ng]
        inj[i, sl["gen_vm"]] = (r[2 * nl + ng:] / gm_full.prod_pu_to_kv).astype(np.float32)   # float32 division, pPB:927
    topo = np.tile(gm_full.default_topo(), (n, 1))
    out, status, iters, busv = eng.run(topo, inj, want_busv=True)
    assert (status == 0).all()
    np.savez_compressed(os.path.join(HERE, "oracle_case14_steps.npz"), scen=scen, rows=rows, inj=inj, topo=topo,
                        out=out, busv=busv, iters=iters)


def case5_chronics():
    """all 20 scenarios of rte_case5_example through the package's own chronics reader (backend order)."""
    from grid2op_b200.chronics import load_scenarios
    env = "rte_case5_example"
    gm = GridModel(os.path.join(REF, env, "grid.json"))
    chron = load_scenarios(os.path.join(REF, env, "chronics"), gm)
    np.savez_compressed(os.path.join(HERE, "case5_chronics.npz"), chron=chron)
    return chron


DATA_TEST_FILES = [
    # what the reference's EXTENDED backend suites (grid2op/_create_test_suite.py with extended_test=True:
    # BaseBackendTest.py goldens :258-319, :438-530, :944-1302, :1584-1670 ...) open under grid2op/data_test — found with an
    # audit hook on `open` while running them; committed so that the suites also run where only the pip-installed
    # reference (no data_test) exists, i.e. on the GPU box
    "test_PandaPower/test_case14.json", "test_PandaPower/prods_charac.csv",
    "chronics/hazards.zip", "chronics/load_p.zip", "chronics/load_q.zip", "chronics/maintenance.zip", "chronics/prod_p.zip",
    "chronics/prod_v.zip",
    "5bus_example_diff_name/config.py", "5bus_example_diff_name/grid.json", "5bus_example_diff_name/grid_layout.json",
    "5bus_example_diff_name/parameters.json", "5bus_example_diff_name/prods_charac.csv",
] + ["5bus_example_diff_name/chronics/0/" + f + ".csv.bz2" for f in (
    "hazards", "load_p", "load_p_forecasted", "load_q", "load_q_forecasted", "maintenance", "prod_p", "prod_p_forecasted", "prod_v",
    "prod_v_forecasted")]


def data_test_fixtures():
    """-> tests/golden/data_test.tar.gz (unpacked on demand by tests/test_backend_suites.py)"""
    import io
    import tarfile
    src_root = os.path.join(os.path.dirname(REF), "data_test")
    with tarfile.open(os.path.join(HERE, "data_test.tar.gz"), "w:gz") as tar:
        for rel in DATA_TEST_FILES:
            with open(os.path.join(src_root, rel), "rb") as f:
                data = f.read()
            info = tarfile.TarInfo("data_test/" + rel)
            info.size = len(data); info.mtime = 0; info.mode = 0o644
            tar.addfile(info, io.BytesIO(data))
    return len(DATA_TEST_FILES)


def env_chronics(env, out_name):
    """every scenario of a bundled environment through the package's own chronics reader (backend order, float32)"""
    from grid2op_b200.chronics import load_scenarios
    gm = GridModel(os.path.join(REF, env, "grid.json"))
    chron = load_scenarios(os.path.join(REF, env, "chronics"), gm)
    np.savez_compressed(os.path.join(HERE, out_name), chron=chron)
    return chron


def simulate_forecast_fixture():
    """-> simulate_forecast_case14.npz: rho of obs.simulate(do_nothing) of unmodified l2rpn_case14_sandbox environments
    (the oracle's PandaPowerBackend restatement solving) behind reset and the first steps of the 3 bundled scenarios, with the
    forecast rows the batched what-if reads for those steps (tests/test_simulate_forecast_gpu.py)"""
    sys.path.insert(0, os.path.dirname(HERE))
    import grid2op_b200.backend as bk
    from grid2op_b200.chronics import _open, list_scenarios, load_forecasts, load_scenarios
    from oracle_engine import OracleEngine
    from test_simulate_forecast_gpu import N_STEPS, obs_simulate_rho

    class OracleBackend(bk.B200Backend):
        def _make_engine(self, gm):
            return OracleEngine(gm)

    env = "l2rpn_case14_sandbox"
    gm = GridModel(os.path.join(REF, env, "grid.json"))
    folders = list_scenarios(os.path.join(REF, env, "chronics"))
    stored = np.load(os.path.join(HERE, "case14_sandbox_chronics.npz"))["chron"]
    assert np.array_equal(load_scenarios(os.path.join(REF, env, "chronics"), gm), stored)
    fc = np.stack([load_forecasts(f, gm)[:N_STEPS] for f in folders])
    has_pv = _open(os.path.join(folders[0], "prod_v_forecasted")) is not None
    want, th = obs_simulate_rho(OracleBackend, len(folders))
    np.savez_compressed(os.path.join(HERE, "simulate_forecast_case14.npz"), want=want, th=th, fc=fc, has_pv=has_pv)
    return want.shape


if __name__ == "__main__":
    print("simulate forecast", simulate_forecast_fixture())
    print("data_test fixtures", data_test_fixtures())
    print("wcci chronics", env_chronics("l2rpn_wcci_2022_dev", "wcci_2022_dev_chronics.npz").shape)
    print("neurips track1 chronics", env_chronics("l2rpn_neurips_2020_track1", "neurips_2020_track1_chronics.npz").shape)
    print("case5 chronics", case5_chronics().shape)
    stored_results()
    gm, chron = case14_chronics()
    print("chronics", chron.shape, chron.dtype)
    grid_models()
    oracle_steps(gm, chron)
