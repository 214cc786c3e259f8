"""The reference's OWN test modules (``grid2op/tests/test_*.py``, unmodified, from the reference tree) with ``B200Backend`` standing
where they expect ``PandaPowerBackend`` (tests/ref_modules_runner.py): environment-, runner-, simulator-, observation- and
rule-level regression tests that exercise the backend through the public API.  CPU: the backend's host logic over the oracle
adapter.  A run over ALL 192 modules of the reference is summarised in ``profiles/round2_reference_test_modules.json`` (133 modules
fully green, 3443 tests run; the rest reach into PandaPowerBackend's private pandapower grid, need gymnasium / matplotlib / the network, or compare
class names that contain "PandaPowerBackend"); this file keeps a curated, fast subset in the suite."""
import json
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))

# (backend-facing modules, each a few seconds at most)
MODULES = [
    # backend behaviour through the env
    "test_dc_isolated_elements", "test_detached_simulate", "test_detached_properly_updated", "test_simulate_disco_load",
    "test_simenv_blackout", "test_no_backend_copy", "test_backend_shunt_deactivated", "test_kirchhoff_obs", "test_simulator",
    "test_soft_overflows", "test_soft_overflow_threshold", "test_remove_line_status_from_topo", "test_back_to_orig",
    "test_previous_state", "test_shedding", "test_issue_sim2real_storage", "test_nb_simulate_called", "test_multi_steps_env",
    "test_redisp_extreme", "test_attached_envs_compat", "test_runner_kwargs_backend", "test_Curtailment", "test_limit_curtail",
    "test_RedispatchEnv", "test_change_param_from_obs", "test_get_info_method", "test_GridGraphObs", "test_elements_graph",
    "test_highres_sim_counter", "test_forecast_from_arrays", "test_multi_steps_forecasts", "test_resest_options",
    # runner / stored episodes
    "test_RunnerFast", "test_EpisodeData", "test_CompactEpisodeData",
    # regression tests of reported issues that go through a power flow
    "test_issue_126", "test_issue_131", "test_issue_146", "test_issue_147", "test_issue_148", "test_issue_151", "test_issue_153",
    "test_issue_164", "test_issue_224", "test_issue_235", "test_issue_245", "test_issue_274", "test_issue_285", "test_issue_319",
    "test_issue_321", "test_issue_327", "test_issue_340", "test_issue_361", "test_issue_364", "test_issue_367", "test_issue_369",
    "test_issue_389", "test_issue_494", "test_issue_503", "test_issue_511", "test_issue_527", "test_issue_538", "test_issue_550",
    "test_issue_591", "test_issue_593", "test_issue_598", "test_issue_616", "test_issue_667", "test_issue_713", "test_issue_731",
    "test_issue_752", "test_issue_redisp_failed_not_illegal",
]


def _run_modules():
    r = subprocess.run([sys.executable, os.path.join(HERE, "ref_modules_runner.py"), "hostlogic"] + MODULES, cwd=HERE, env=dict(os.environ),
                       capture_output=True, text=True, timeout=1500)
    out = {}
    for ln in r.stdout.splitlines():
        if ln.startswith("RESULT "):
            d = json.loads(ln[7:])
            out[d["module"]] = d
    if not out:
        pytest.fail("runner produced nothing: " + r.stderr[-1500:])
    return out


@pytest.fixture(scope="module")
def results(request, tmp_path_factory):
    from conftest import grid2op_root
    root = grid2op_root()
    if root is None or not os.path.isdir(os.path.join(root, "tests")) or not os.path.isdir(os.path.join(root, "data_test")):
        pytest.skip("reference test tree (with its data_test fixtures) not available")
    uid = getattr(request.config, "workerinput", {}).get("testrunuid")
    if uid is None:                      # plain (serial) run
        return _run_modules()
    # pytest-xdist: every worker that receives one of the parametrised tests would run the modules again — concurrently, and
    # some of them write into shared scratch directories of the reference tree.  One worker runs them, the others read its result.
    import fcntl
    path = os.path.join(str(tmp_path_factory.getbasetemp().parent), f"reference_modules_{uid}.json")
    with open(path + ".lock", "w") as lock:
        fcntl.flock(lock, fcntl.LOCK_EX)
        if os.path.exists(path):
            with open(path) as f:
                return json.load(f)
        out = _run_modules()
        with open(path, "w") as f:
            json.dump(out, f)
        return out


@pytest.mark.parametrize("module", MODULES)
def test_reference_module_green_on_b200_backend(results, module):
    d = results.get(module)
    assert d is not None, f"{module}: no result (the runner stopped before it)"
    assert "import_error" not in d, d
    assert d["run"] > 0 and d["fail"] == 0 and d["err"] == 0, d
