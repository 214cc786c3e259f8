"""TEST INFRASTRUCTURE: ctypes front-end of tests/emu/sparse_emu.cpp (host build of the planned sparse kernel)."""
from __future__ import annotations

import ctypes as C
import os
import subprocess

import numpy as np

HERE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "emu")
REPO = os.path.dirname(os.path.dirname(HERE))
LIB = os.path.join(HERE, "libsparse_emu.so")


def build(force: bool = False) -> str:
    src = os.path.join(HERE, "sparse_emu.cpp")
    deps = [src] + [os.path.join(REPO, "grid2op_b200", "csrc", f) for f in ("b200pf_sparse.cuh", "b200pf_plan.hpp", "b200pf_block.cuh")]
    if force or not os.path.exists(LIB) or os.path.getmtime(LIB) < max(os.path.getmtime(p) for p in deps):
        # compiled under a private name and renamed into place: parallel test workers may build it at the same time
        tmp = f"{LIB}.{os.getpid()}.tmp"
        subprocess.check_call(["g++", "-O2", "-std=c++17", "-fPIC", "-shared", "-x", "c++", "-o", tmp, src, "-lm"])
        os.replace(tmp, LIB)
    return LIB


class SparseEmu:
    """Same call signature as oracle.c_oracle.COracle.run / PowerFlowEngine.run."""

    def __init__(self, gm):
        from oracle.c_oracle import COracle
        build()
        self.gm = gm
        self._co = COracle(gm)          # re-use its grid descriptor marshalling
        self.desc = self._co.desc
        self.lib = C.CDLL(LIB)
        self.lib.sparse_emu_run.restype = C.c_int
        self.stats = np.zeros(8, dtype=np.int32)

    def run(self, topo, inj, is_dc=False, max_iter=10, tol_mva=1e-8, nb_cap=0, want_busv=False, n1_lines=0, th_lim=None):
        gm = self.gm
        topo = np.ascontiguousarray(topo, dtype=np.int8).reshape(-1, gm.n_topo_in)
        inj = np.ascontiguousarray(inj, dtype=np.float64).reshape(-1, gm.n_inj)
        B = topo.shape[0]
        N = B * n1_lines if n1_lines > 0 else B
        out = np.empty((N, gm.n_out), dtype=np.float32)
        status = np.empty(N, dtype=np.int32)
        iters = np.empty(N, dtype=np.int32)
        busv = np.empty((N, 2 * gm.n_sub * gm.n_busbar), dtype=np.float64) if want_busv else None
        rho = np.empty((N, gm.n_line), dtype=np.float32) if th_lim is not None else None
        thl = np.ascontiguousarray(th_lim, dtype=np.float32) if th_lim is not None else None
        vp = C.c_void_p
        self.lib.sparse_emu_run(C.byref(self.desc), C.c_int(B), topo.ctypes.data_as(vp), inj.ctypes.data_as(vp),
                                C.c_int(int(bool(is_dc))), C.c_int(int(max_iter)), C.c_double(float(tol_mva)),
                                out.ctypes.data_as(vp), status.ctypes.data_as(vp), iters.ctypes.data_as(vp),
                                busv.ctypes.data_as(vp) if busv is not None else None, C.c_int(int(n1_lines)),
                                thl.ctypes.data_as(vp) if thl is not None else None,
                                rho.ctypes.data_as(vp) if rho is not None else None, self.stats.ctypes.data_as(vp))
        if th_lim is not None:
            return out, status, iters, busv, rho
        return out, status, iters, busv


class BlockEmu(SparseEmu):
    """Host build of the BLOCK-planned kernel (csrc/b200pf_block.cuh) with T lanes per instance, U operations per lane and row."""

    def __init__(self, gm, T=4, U=2):
        super().__init__(gm)
        self.T, self.U = int(T), int(U)
        self.lib.block_emu_run.restype = C.c_int

    def run(self, topo, inj, is_dc=False, max_iter=10, tol_mva=1e-8, nb_cap=0, want_busv=False, n1_lines=0, th_lim=None):
        gm = self.gm
        topo = np.ascontiguousarray(topo, dtype=np.int8).reshape(-1, gm.n_topo_in)
        inj = np.ascontiguousarray(inj, dtype=np.float64).reshape(-1, gm.n_inj)
        B = topo.shape[0]
        N = B * n1_lines if n1_lines > 0 else B
        out = np.empty((N, gm.n_out), dtype=np.float32)
        status = np.empty(N, dtype=np.int32)
        iters = np.empty(N, dtype=np.int32)
        busv = np.empty((N, 2 * gm.n_sub * gm.n_busbar), dtype=np.float64) if want_busv else None
        rho = np.empty((N, gm.n_line), dtype=np.float32) if th_lim is not None else None
        thl = np.ascontiguousarray(th_lim, dtype=np.float32) if th_lim is not None else None
        vp = C.c_void_p
        rc = self.lib.block_emu_run(C.byref(self.desc), C.c_int(self.T), C.c_int(self.U), C.c_int(B), topo.ctypes.data_as(vp),
                                    inj.ctypes.data_as(vp), C.c_int(int(bool(is_dc))), C.c_int(int(max_iter)), C.c_double(float(tol_mva)),
                                    out.ctypes.data_as(vp), status.ctypes.data_as(vp), iters.ctypes.data_as(vp),
                                    busv.ctypes.data_as(vp) if busv is not None else None, C.c_int(int(n1_lines)),
                                    thl.ctypes.data_as(vp) if thl is not None else None,
                                    rho.ctypes.data_as(vp) if rho is not None else None, self.stats.ctypes.data_as(vp))
        assert rc == 0, rc
        if th_lim is not None:
            return out, status, iters, busv, rho
        return out, status, iters, busv


def validate_block_plan(gm, topo_row, outage=-1, T=4, U=2):
    """-> (return code of block_emu_validate_plan, residual, [nblk, passes, rows, smem bytes per instance, real operations])"""
    emu = SparseEmu(gm)
    err = C.c_double(0.0)
    info = np.zeros(8, dtype=np.int32)
    t = np.ascontiguousarray(topo_row, dtype=np.int8)
    emu.lib.block_emu_validate_plan.restype = C.c_int
    rc = emu.lib.block_emu_validate_plan(C.byref(emu.desc), t.ctypes.data_as(C.c_void_p), C.c_int(int(outage)), C.c_int(int(T)), C.c_int(int(U)),
                                         C.byref(err), info.ctypes.data_as(C.c_void_p))
    return int(rc), float(err.value), info[:5].tolist()


def validate_plan(gm, topo_row, outage=-1, op_width=32):
    """-> (return code of sparse_emu_validate_plan, residual of A x = b through the operation stream)."""
    emu = SparseEmu(gm)
    err = C.c_double(0.0)
    t = np.ascontiguousarray(topo_row, dtype=np.int8)
    emu.lib.sparse_emu_validate_plan.restype = C.c_int
    rc = emu.lib.sparse_emu_validate_plan(C.byref(emu.desc), t.ctypes.data_as(C.c_void_p), C.c_int(int(outage)), C.c_int(int(op_width)),
                                          C.byref(err))
    return int(rc), float(err.value)


class EmuProtRollout:
    """Batched DoNothing rollout with protections through the emulated planned kernel + the host cascade loop
    (tests/emu/sparse_emu.cpp: sparse_emu_series_prot_step), state held in numpy arrays."""

    def __init__(self, gm, chron, scen, t0, thermal_limit_a, hard=2.0, soft=1.0, max_allowed=2):
        self.emu = SparseEmu(gm)
        self.gm = gm
        self.chron = np.ascontiguousarray(chron, dtype=np.float32)
        self.B = len(scen)
        self.scen = np.ascontiguousarray(scen, dtype=np.int32)
        self.t = np.ascontiguousarray(t0, dtype=np.int32).copy()
        self.topo = np.ascontiguousarray(np.tile(gm.default_topo(), (self.B, 1)), dtype=np.int8)
        self.static_inj = np.ascontiguousarray(gm.default_inj(), dtype=np.float64)
        self.th = np.ascontiguousarray(thermal_limit_a, dtype=np.float32)
        self.hard, self.soft, self.max_allowed = float(hard), float(soft), int(max_allowed)
        nl = gm.n_line
        self.out = np.zeros((self.B, gm.n_out), dtype=np.float32)
        self.status = np.zeros(self.B, dtype=np.int32)
        self.iters = np.zeros(self.B, dtype=np.int32)
        self.rho = np.zeros((self.B, nl), dtype=np.float32)
        self.pcount = np.zeros((self.B, nl), dtype=np.int32)
        self.ts_over = np.zeros((self.B, nl), dtype=np.int32)
        self.disc = np.full((self.B, nl), -1, dtype=np.int32)
        self.done = np.zeros(self.B, dtype=np.int32)
        self.rounds = np.zeros(1, dtype=np.int32)
        self.emu.lib.sparse_emu_series_prot_step.restype = C.c_int

    def step(self, from_reset=False):
        vp = C.c_void_p
        p = lambda a: a.ctypes.data_as(vp)     # noqa: E731
        rc = self.emu.lib.sparse_emu_series_prot_step(
            C.byref(self.emu.desc), C.c_int(self.B), p(self.topo), p(self.chron), C.c_int(self.chron.shape[0]), C.c_int(self.chron.shape[1]),
            p(self.scen), p(self.t), p(self.static_inj), p(self.th), C.c_int(int(from_reset)), C.c_float(self.hard), C.c_float(self.soft),
            C.c_int(self.max_allowed), C.c_int(10), C.c_double(1e-8), p(self.out), p(self.status), p(self.iters), p(self.rho),
            p(self.pcount), p(self.ts_over), p(self.disc), p(self.done), p(self.rounds))
        assert rc == 0, rc
        return int(self.rounds[0])
