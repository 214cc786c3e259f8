"""Batched ``obs.simulate`` on forecasts (``BatchedDoNothing.simulate_forecast``: one launch for the what-if of every
instance) against ``obs.simulate(do_nothing)`` of unmodified grid2op environments on l2rpn_case14_sandbox
(reference grid2op/Observation/baseObservation.py:3365-3669, forecasts from GridStateFromFileWithForecasts).

What those environments compute is stored in ``tests/golden/simulate_forecast_case14.npz`` (written by
``tests/golden/make_golden.py``), so the GPU test needs neither grid2op nor its bundled data; where both are importable the
tests also step live environments and check that they still compute the stored values."""
import os
import warnings

import numpy as np
import pytest

from conftest import env_grid

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
FIXTURE = os.path.join(GOLD, "simulate_forecast_case14.npz")
N_STEPS = 5


def obs_simulate_rho(backend_factory, n_scen, n_steps=N_STEPS):
    """rho of ``obs.simulate(do_nothing)`` after reset and after each of the first steps of every bundled scenario of an
    unmodified l2rpn_case14_sandbox environment -> (float32 [n_scen, n_steps, n_line], thermal limits)"""
    import grid2op_b200.backend  # noqa: F401  (locates the grid2op install)
    import grid2op
    from grid2op.Parameters import Parameters
    p = Parameters()
    p.NO_OVERFLOW_DISCONNECTION = True
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        env = grid2op.make("l2rpn_case14_sandbox", test=True, backend=backend_factory(), param=p, _add_to_name="simfc" + backend_factory.__name__)
    th = np.asarray(env.get_thermal_limit(), dtype=np.float32)
    want = np.zeros((n_scen, n_steps, env.n_line), dtype=np.float32)
    for sc in range(n_scen):
        env.set_id(sc)
        obs = env.reset()
        for k in range(n_steps):
            sim, _, done, info = obs.simulate(env.action_space())
            assert not done, info["exception"]
            want[sc, k] = sim.rho
            obs, _, done, _ = env.step(env.action_space())
            assert not done
    env.close()
    return want, th


def batched_rho(gm, chron, fc, has_pv, th, engine, n_steps=N_STEPS):
    """``simulate_forecast`` behind each of the first steps of a BatchedDoNothing with one instance per scenario
    -> float32 [n_scen, n_steps, n_line]"""
    from grid2op_b200.rollout import BatchedDoNothing
    n_scen = chron.shape[0]
    benv = BatchedDoNothing(gm, chron, n_scen, scen=np.arange(n_scen), t0=np.zeros(n_scen), thermal_limit_a=th, engine=engine)
    got = np.zeros((n_scen, n_steps, gm.n_line), dtype=np.float32)
    for k in range(n_steps):
        benv.step_device()                                   # the step the environment has done (reset = row 0, then one per step)
        benv.fetch()
        out, status, rho = benv.simulate_forecast(fc, forecast_has_prod_v=has_pv)
        assert (status == 0).all()
        got[:, k] = rho
    benv.close()
    return got


def _check(got, want, what):
    assert np.allclose(got, want, rtol=2e-4, atol=2e-5), (what, float(np.max(np.abs(got - want))))


def _run(backend_factory, engine_factory):
    grid = env_grid("l2rpn_case14_sandbox")
    if grid is None:
        pytest.skip("reference data not available")
    import grid2op_b200.backend  # noqa: F401  (locates the grid2op install)
    from grid2op_b200.chronics import _open, list_scenarios, load_forecasts, load_scenarios
    from grid2op_b200.gridmodel import GridModel
    gm = GridModel(grid)
    cdir = os.path.join(os.path.dirname(grid), "chronics")
    folders = list_scenarios(cdir)
    chron = load_scenarios(cdir, gm)
    fc = np.stack([load_forecasts(f, gm) for f in folders])
    has_pv = _open(os.path.join(folders[0], "prod_v_forecasted")) is not None
    want, th = obs_simulate_rho(backend_factory, len(folders))
    _check(batched_rho(gm, chron, fc, has_pv, th, engine_factory(gm)), want, "live environments")
    z = np.load(FIXTURE)
    _check(want, z["want"], "stored fixture")


@pytest.mark.gpu
def test_batched_simulate_on_forecasts_matches_obs_simulate(cuda_required):
    from grid2op_b200._bootstrap import ensure_grid2op
    from grid2op_b200.gridmodel import GridModel
    gm = GridModel.from_npz(os.path.join(GOLD, "gridmodel_l2rpn_case14_sandbox.npz"))
    chron = np.load(os.path.join(GOLD, "case14_sandbox_chronics.npz"))["chron"]
    z = np.load(FIXTURE)
    _check(batched_rho(gm, chron, z["fc"], bool(z["has_pv"]), z["th"], None), z["want"], "stored obs.simulate")
    if env_grid("l2rpn_case14_sandbox") is not None and ensure_grid2op():
        from grid2op_b200.backend import B200Backend
        _run(B200Backend, lambda gm: None)


def test_batched_simulate_on_forecasts_host_logic():
    """CPU counterpart: which forecast row belongs to which step, voltage set points without a prod_v forecast — reference
    environments on the oracle adapter, the batched driver on the oracle's C restatement (test infrastructure)"""
    if env_grid("l2rpn_case14_sandbox") is None:
        pytest.skip("reference data not available")
    import grid2op_b200.backend as bk
    from oracle_engine import COracleSeriesEngine, OracleEngine

    class HostLogicBackendSim(bk.B200Backend):
        def _make_engine(self, gm):
            return OracleEngine(gm)

    _run(HostLogicBackendSim, COracleSeriesEngine)
