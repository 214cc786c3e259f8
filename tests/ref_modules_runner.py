"""TEST INFRASTRUCTURE.  Runs test modules of the reference (``grid2op/tests/test_*.py``, unmodified) with ``B200Backend`` standing
where they expect ``PandaPowerBackend`` — the default backend of ``grid2op.make`` (the environments' ``config.py`` take it from
``grid2op.Backend``), of the Runner, and of tests that name it — and prints one JSON line per module:

    python tests/ref_modules_runner.py hostlogic|gpu module [module ...]

``hostlogic``: the backend's host code over the oracle adapter (no GPU); ``gpu``: the CUDA engine.  Tests that reach into
PandaPowerBackend's private pandapower grid (``backend._grid``), or that need packages this image does not have (gymnasium,
matplotlib, lightsim2grid), cannot pass by construction and are not in the curated list of tests/test_reference_modules.py.
"""
import importlib
import json
import os
import sys
import time
import types
import unittest
import warnings

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE)); sys.path.insert(0, HERE)


import conftest  # noqa: F401,E402
import grid2op_b200.backend as bk  # noqa: E402


class HostLogicStand(bk.B200Backend):
    """(module level: the reference's multi-process runner tests pickle the backend class)"""

    def _make_engine(self, gm):
        from oracle_engine import OracleEngine
        return OracleEngine(gm)


def main():
    mode, mods = sys.argv[1], sys.argv[2:]
    Stand = HostLogicStand if mode == "hostlogic" else bk.B200Backend
    import grid2op  # noqa: F401
    import grid2op.Backend as GB
    import grid2op.Backend.pandaPowerBackend as GBP
    import grid2op.MakeEnv.MakeFromPath as MFP
    import grid2op.Runner.runner as RR
    for m in (GB, GBP, MFP, RR):
        m.PandaPowerBackend = Stand
    if "lightsim2grid" not in sys.modules:          # some modules import it for a variant of their tests
        ls = types.ModuleType("lightsim2grid"); ls.LightSimBackend = Stand; sys.modules["lightsim2grid"] = ls
    for name in mods:
        out = {"module": name}
        t0 = time.time()
        try:
            with warnings.catch_warnings():
                warnings.simplefilter("ignore")
                mod = importlib.import_module("grid2op.tests." + name)
                suite = unittest.defaultTestLoader.loadTestsFromModule(mod)
                with open(os.devnull, "w") as sink:
                    res = unittest.TextTestRunner(verbosity=0, stream=sink).run(suite)
            out.update(run=res.testsRun, fail=len(res.failures), err=len(res.errors), skip=len(res.skipped),
                       bad=[(t.id().split(".", 3)[-1], tb.strip().splitlines()[-1][:200]) for t, tb in (res.failures + res.errors)[:10]])
        except BaseException as exc:  # noqa: BLE001
            out.update(import_error=repr(exc)[:300])
        out["sec"] = round(time.time() - t0, 1)
        print("RESULT " + json.dumps(out), flush=True)


if __name__ == "__main__":
    main()
