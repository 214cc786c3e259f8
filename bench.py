#!/usr/bin/env python
"""bench.py - env.step()/s of the batched power-flow hot path (BASELINE.json metric).

    python bench.py --gpus N --steps K --warmup W            # our CUDA path (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K ...  # CPU arm: the oracle's C restatement on the host cores
    python bench.py --workload wcci --gpus N ...             # BASELINE.json configs[4]: 118 substations, batch 8192 in total
    python bench.py ... --dump-outputs DIR                   # + the last timed step's results as DIR/<name>.npy (float32)

Workload `case14` (default; BASELINE.json configs[1], the configuration the metric is quoted on): l2rpn_case14_sandbox, AC
Newton-Raphson, batch 4096 per GPU (weak scaling), DoNothing rollout over the bundled chronics (instance i -> scenario i mod 3,
start row (i*37) mod 576; SURVEY.md 8(d)), NO_OVERFLOW_DISCONNECTION like the reference's own profiling script.
Workload `wcci` (configs[4]): l2rpn_wcci_2022 (= grid2op/data/l2rpn_wcci_2022_dev, 118 substations), AC, batch 8192 IN TOTAL
sharded over the N GPUs (strong scaling), DoNothing over the bundled 289-row scenario.
A "step" is one pass of the hot path over the whole batch = batch env.step() calls.

N > 1: independent instances, no collective inside the solve.  The step results every rank owes the agent's rank (rho, 4 bytes
per line and instance) go into a device ring of 2 x 64 step slots; ONE NCCL gather per 64 steps ships a half ring to rank 0,
asynchronously, while the kernels fill the other half (measured on 2 x B200: 0.98 weak-scaling efficiency).  `--collect p2p`
is the alternative without any collective: the kernels store rho AND a per-rank completion word straight into rank 0's HBM
through a peer mapping over NVLink (CUDA IPC, include/b200pf.h "Multi-GPU result collection"); it measured slower (0.88-0.91:
the remote stores and their system-wide fence sit on the step's critical path), so it is the option, not the default.

One JSON line on stdout (rank 0).  Keys documented in DESIGN.md section "Measurement".
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

REPO = os.path.dirname(os.path.abspath(__file__))
if REPO not in sys.path:
    sys.path.insert(0, REPO)
GOLD = os.path.join(REPO, "tests", "golden")

UNIT = "env.step()/s"
WORKLOADS = {
    "case14": dict(metric="env.step()/sec at batch on l2rpn_case14 AC", env="l2rpn_case14_sandbox",
                   grid="gridmodel_l2rpn_case14_sandbox.npz", chron="case14_sandbox_chronics.npz", batch_per_gpu=4096,
                   total_batch=None, scaling="weak"),
    "wcci": dict(metric="env.step()/sec at batch on l2rpn_wcci_2022 AC", env="l2rpn_wcci_2022 (l2rpn_wcci_2022_dev, 118 substations)",
                 grid="gridmodel_l2rpn_wcci_2022_dev.npz", chron="wcci_2022_dev_chronics.npz", batch_per_gpu=None,
                 total_batch=8192, scaling="strong"),
}


def load_workload(name="case14"):
    from grid2op_b200.gridmodel import GridModel
    w = WORKLOADS[name]
    gm = GridModel.from_npz(os.path.join(GOLD, w["grid"]))
    chron = np.load(os.path.join(GOLD, w["chron"]))["chron"]
    return gm, chron


def nr_dimension(gm):
    n_ref = 1
    n_pv = int(len(set(int(x) for x in gm.gen_sub))) - n_ref
    return n_pv + 2 * (gm.n_sub - n_pv - n_ref)


def flops_view(gm, mean_iters, batch, kern_s, clocks):
    """SURVEY.md 8(d), second view: dense-LU flops per instance-iteration (2/3 d^3 + 2 d^2, d = NR dimension with all
    elements on busbar 1) against the fp32 CUDA-core peak at the SM clock sampled during the run (148 SMs x 128 FMA
    lanes x 2; the per-instance systems are far too small and sparse for tensor cores, so MEASURED_PEAKS' bf16 figure
    does not apply).  The planned kernels do the SPARSE factorisation, i.e. far fewer flops than this view credits."""
    d = nr_dimension(gm)
    fl = (2.0 / 3.0) * d ** 3 + 2.0 * d ** 2
    ach = batch * fl * mean_iters / kern_s / 1e12
    mhz = (clocks or {}).get("sm_mhz") or 1965
    peak = 148 * 128 * 2 * mhz * 1e6 / 1e12
    return {"nr_dimension": d, "flops_per_instance_iteration": fl, "achieved_tflops": ach, "peak_fp32_cuda_core_tflops": peak,
            "frac": ach / peak}


def measured_peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def algorithmic_bytes(gm, mean_iters):
    """SURVEY.md 8(d): B_iter (state round-tripped through HBM once per NR iteration, int8 topo, fp64
    V as we keep it) x iterations + result write-back.  Also the compulsory bytes of THIS design (fused:
    inputs read once, results written once)."""
    n_bus_max = gm.n_slot
    inj_vals = 2 * gm.n_load + 2 * gm.n_gen + gm.n_storage + 3 * gm.n_shunt
    b_iter = gm.dim_topo + 4 * inj_vals + 2 * 16 * n_bus_max + 4
    result = 4 * gm.n_out
    survey = b_iter * mean_iters + result
    compulsory = 4 * (2 * gm.n_load + 2 * gm.n_gen) + gm.n_topo_in + 8 + 4 * gm.n_out + 4 * gm.n_line + 8
    return float(survey), float(compulsory), int(b_iter)


def profiled_traffic(kernel_tag):
    """dram bytes per launch of the dominant kernel from the newest committed `ncu --set full` summary whose kernel tag equals
    the kernel this run launched; None when no such profile exists (a stale number is worse than none)."""
    pdir = os.path.join(REPO, "profiles")
    best = None
    try:
        for fn in sorted(os.listdir(pdir)):
            if not (fn.endswith("_summary.json") and "ncu" in fn):
                continue
            try:
                d = json.load(open(os.path.join(pdir, fn)))
            except Exception:
                continue
            if d.get("kernel_tag") == kernel_tag and d.get("dram_bytes_per_launch") is not None:
                best = (d["dram_bytes_per_launch"], fn)
    except OSError:
        pass
    return best


class ClockSampler(threading.Thread):
    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self._halt = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._halt.is_set():
            try:
                o = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                   capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            self._halt.wait(0.1)

    def stop(self):
        self._halt.set()
        self.join(timeout=6)
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": float(max(mx)) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------------------------
# CPU arm
# ---------------------------------------------------------------------------------------------------------------
def host_cpu_info():
    """logical CPUs this process may run on, physical cores among them, and the cgroup CPU quota (None = unlimited)"""
    try:
        aff = sorted(os.sched_getaffinity(0))
    except Exception:
        aff = list(range(os.cpu_count() or 1))
    cores = set()
    try:
        phys, core, proc = None, None, None
        for line in open("/proc/cpuinfo"):
            if line.startswith("processor"):
                proc = int(line.split(":")[1])
            elif line.startswith("physical id"):
                phys = int(line.split(":")[1])
            elif line.startswith("core id"):
                core = int(line.split(":")[1])
            elif not line.strip():
                if proc in aff and core is not None:
                    cores.add((phys, core))
                phys = core = proc = None
    except Exception:
        pass
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        pass
    return {"logical": len(aff), "physical": len(cores) or len(aff), "cgroup_quota_cpus": quota}


def _pin_openmp():
    # must happen before libgomp is loaded (the first COracle): threads stay on their cores, spin instead of sleeping
    os.environ.setdefault("OMP_PROC_BIND", "close")
    os.environ.setdefault("OMP_PLACES", "cores")
    os.environ.setdefault("OMP_WAIT_POLICY", "active")
    os.environ.pop("OMP_NUM_THREADS", None)           # torchrun exports OMP_NUM_THREADS=1; the arm sets its count explicitly


class CpuArm:
    """oracle/pf_oracle.c (fp64 dense Newton, OpenMP over instances) stepping the same DoNothing workload."""

    def __init__(self, gm, chron, n_inst):
        from oracle.c_oracle import COracle
        from grid2op_b200.rollout import instance_schedule
        self.COracle = COracle
        self.gm, self.chron, self.n = gm, chron, n_inst
        self.scen, self.t0 = instance_schedule(n_inst, chron.shape[0], chron.shape[1])
        self.sl = gm.inj_slices()
        self.topo = np.tile(gm.default_topo(), (n_inst, 1))
        self.inj = np.tile(gm.default_inj(), (n_inst, 1))
        self.info = host_cpu_info()
        self.orc = None
        self.nthreads = 0

    def _fill(self, k):
        gm, sl, nl, ng = self.gm, self.sl, self.gm.n_load, self.gm.n_gen
        rows = self.chron[self.scen, (self.t0 + k) % self.chron.shape[1]]
        self.inj[:, sl["load_p"]] = rows[:, :nl]; self.inj[:, sl["load_q"]] = rows[:, nl:2 * nl]
        self.inj[:, sl["gen_p"]] = rows[:, 2 * nl:2 * nl + ng]
        self.inj[:, sl["gen_vm"]] = rows[:, 2 * nl + ng:] / gm.prod_pu_to_kv[None, :]

    def calibrate(self):
        """thread count: logical CPUs, physical cores, the cgroup quota - whichever steps the batch fastest (>= 0.3 s each)"""
        info = self.info
        cands = {info["logical"], info["physical"]}
        if info["cgroup_quota_cpus"]:
            cands.add(max(1, int(round(info["cgroup_quota_cpus"]))))
        best = None
        self._fill(0)
        for nt in sorted(c for c in cands if c >= 1):
            o = self.COracle(self.gm, nthreads=nt)
            o.run(self.topo, self.inj)
            t, reps = time.perf_counter(), 0
            while time.perf_counter() - t < 0.3:
                o.run(self.topo, self.inj); reps += 1
            rate = reps * self.n / (time.perf_counter() - t)
            if best is None or rate > best[0]:
                best = (rate, nt, o)
        self.orc, self.nthreads = best[2], best[1]

    def step(self, k):
        self._fill(k)
        t = time.perf_counter()
        out, status, iters, _ = self.orc.run(self.topo, self.inj)
        dt = time.perf_counter() - t
        assert (status == 0).all()
        self.last = (out, status, iters)
        return dt

    def sample(self, min_steps, min_seconds, warmup=2):
        """-> per-step solver times (the host-side row gather is not counted, like the GPU arm's resident inputs)"""
        if self.orc is None:
            self.calibrate()
        for k in range(warmup):
            self.step(k)
        ts, k = [], warmup
        while len(ts) < min_steps or sum(ts) < min_seconds:
            ts.append(self.step(k)); k += 1
        return np.array(ts)

    def describe(self, ts):
        info = self.info
        return (f"{len(ts)} steps x {self.n} instances in {ts.sum():.1f} s, oracle/pf_oracle.c (fp64 dense Newton), OpenMP x{self.nthreads} "
                f"pinned (host: {info['logical']} logical / {info['physical']} physical CPUs"
                + (f", cgroup quota {info['cgroup_quota_cpus']:.1f}" if info["cgroup_quota_cpus"] else "") + ")")


def run_reference(args):
    """CPU arm.  The reference's implementation of this path is pandapower (pure Python, third party,
    not installable here - no wheel, no network); the arm therefore times the oracle's C restatement of
    the same algorithm on all host cores: a (much) faster stand-in than the original, labelled 'port'."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    _pin_openmp()
    w = WORKLOADS[args.workload]
    gm, chron = load_workload(args.workload)
    batch = args.batch or (w["batch_per_gpu"] or w["total_batch"])
    arm = CpuArm(gm, chron, batch)
    ts = arm.sample(args.steps, args.cpu_min_seconds, warmup=max(args.warmup, 1))
    if args.dump_outputs:
        from grid2op_b200.engine import OutputView
        out, status, iters = arm.last
        dump_outputs(args.dump_outputs, gm, out, status, iters, OutputView(gm, out).a_or / gm.thermal_limit_a[None, :])
    rates = batch / ts
    value = float(np.median(rates))
    line = {
        "impl": "reference", "metric": w["metric"], "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": int(len(ts)),
        "warmup": max(args.warmup, 1), "ms_per_step": float(1e3 * np.median(ts)), "higher_is_better": True, "scaling": w["scaling"],
        "vs_baseline": None, "dtype": "f64", "data": f"synthetic (bundled {w['env']} chronics rows replayed, DoNothing)",
        # (the same `workload` text as the GPU arm prints for this workload: the two lines describe one configuration)
        "config": {"workload": f"{w['env']} AC Newton-Raphson, batch {batch} envs per GPU, DoNothing rollout", "batch_per_step": batch,
                   "arm": "host CPU: one batch of that size per step, all host threads the cgroup grants",
                   "requested_steps": args.steps,
                   "note": "value = median over the steps of batch / step time; --cpu-min-seconds > 0 adds steps until the arm has run that long"},
        "spread": {"min": float(rates.min()), "median": value, "max": float(rates.max()), "unit": UNIT, "n": int(len(ts))},
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": arm.nthreads, "kind": "port", "sample": arm.describe(ts),
                         "host": arm.info},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, gm, out, status, iters, rho):
    """``--dump-outputs``: what the timed path returned for its last step as ``<dirname>/<name>.npy`` (float32): ``rho``,
    every field of the result record (engine.OutputView) the grid has elements for, the solver ``status`` and Newton
    ``iterations`` per instance.  Above 64 MB in all, a fixed seeded sample of instances is written, their indices in
    ``instance.npy``."""
    from grid2op_b200.engine import OutputView
    idx = np.arange(len(status))
    row_bytes = 4 * (gm.n_out + gm.n_line + 2)
    if len(idx) * row_bytes > DUMP_LIMIT_BYTES:
        n = (DUMP_LIMIT_BYTES - 4096) // (row_bytes + 4)
        idx = np.sort(np.random.default_rng(0).choice(len(idx), n, replace=False))
    view = OutputView(gm, out[idx])
    arrays = {"rho": rho[idx], "status": status[idx], "iterations": iters[idx]}
    arrays.update((name, getattr(view, name)) for name in OutputView.FIELDS)
    if len(idx) < len(status):
        arrays["instance"] = idx
    os.makedirs(dirname, exist_ok=True)
    for name, a in arrays.items():
        if a.size == 0:                 # no element of that kind (e.g. no storage unit on the grid)
            continue
        np.save(os.path.join(dirname, name + ".npy"), np.ascontiguousarray(a, dtype=np.float32))


# ---------------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------------
def parity_sample(gm, chron, env, out, status, n_series_steps, n_sample=256):
    """Self-check of the timed path: the result records of the LAST timed step, for a sample of instances, against the
    fp64 oracle (C restatement) on the same chronics rows.  -> dict; max_err_pu in p.u. (flows / sn_mva, voltages / vn)."""
    from oracle.c_oracle import COracle
    from grid2op_b200.engine import OutputView
    B = env.batch
    idx = np.unique(np.linspace(0, B - 1, min(n_sample, B)).astype(np.int64))
    rows = chron[env.scen[idx], (env.t0[idx].astype(np.int64) + n_series_steps - 1) % chron.shape[1]]
    sl, nl, ng = gm.inj_slices(), gm.n_load, gm.n_gen
    inj = np.tile(gm.default_inj(), (len(idx), 1))
    inj[:, sl["load_p"]] = rows[:, :nl]; inj[:, sl["load_q"]] = rows[:, nl:2 * nl]
    inj[:, sl["gen_p"]] = rows[:, 2 * nl:2 * nl + ng]
    inj[:, sl["gen_vm"]] = (rows[:, 2 * nl + ng:] / gm.prod_pu_to_kv[None, :]).astype(np.float32)
    ref, rstatus, _, _ = COracle(gm).run(np.tile(gm.default_topo(), (len(idx), 1)), inj)
    a, b = OutputView(gm, out[idx]), OutputView(gm, ref)
    err = 0.0
    for k in ("p_or", "q_or", "p_ex", "q_ex", "unit_p", "unit_q"):
        err = max(err, float(np.max(np.abs(getattr(a, k).astype(np.float64) - getattr(b, k)))) / gm.sn_mva)
    for k, vn in (("v_or", gm.line_or_vn), ("v_ex", gm.line_ex_vn), ("load_v", gm.load_vn)):
        err = max(err, float(np.max(np.abs(getattr(a, k).astype(np.float64) - getattr(b, k)) / vn)))
    same_status = bool(np.array_equal(status[idx], rstatus))
    return {"instances": int(len(idx)), "max_err_pu": err, "tolerance_pu": 1e-4, "status_equal": same_status,
            "ok": bool(err < 1e-4 and same_status), "against": "oracle/pf_oracle.c (fp64, partial pivoting) on the same chronics rows"}


def run_ours(args):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - this path has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    from grid2op_b200.collect import RingCollector
    from grid2op_b200.engine import PeerBuffer
    from grid2op_b200.rollout import BatchedDoNothing
    os.environ["B200PF_PLAN_POLICY"] = str(args.policy)
    if args.no_redo:
        os.environ["B200PF_NO_REDO"] = "1"
    w = WORKLOADS[args.workload]
    gm, chron = load_workload(args.workload)
    if args.batch:
        batch = args.batch
    elif w["batch_per_gpu"]:
        batch = w["batch_per_gpu"]
    else:
        batch = w["total_batch"] // world
    env = BatchedDoNothing(gm, chron, batch, device=local, offset=rank * batch)
    eng = env.engine
    stream = torch.cuda.Stream()            # a real (non-default) stream shared by torch events and the engine
    torch.cuda.set_stream(stream)
    eng.set_stream(stream.cuda_stream)
    status = torch.empty((batch,), dtype=torch.int32, device="cuda")
    iters = torch.empty((batch,), dtype=torch.int32, device="cuda")
    nl = gm.n_line
    K = max(1, args.gather_every)
    slot_elems = batch * nl
    # ---- where rho goes: a ring of 2K step slots per rank inside ONE buffer in rank 0's HBM ------------------------------
    # (two halves of K slots: while the kernels fill one half the agent owns the other)
    collect = args.collect if world > 1 else "local"
    peer, ring_local, gather_lists = None, None, None
    ring_bytes = world * 2 * K * slot_elems * 4
    if collect == "p2p":
        ok = 1
        handle = torch.zeros(64, dtype=torch.uint8, device="cuda")
        try:
            if rank == 0:
                peer = PeerBuffer(ring_bytes + 256)           # + one completion word per rank behind the ring
                handle.copy_(torch.frombuffer(bytearray(peer.handle), dtype=torch.uint8))
        except Exception as exc:      # noqa: BLE001
            ok = 0
            print(f"bench.py: peer buffer export failed on rank 0: {exc}", file=sys.stderr)
        dist.broadcast(handle, src=0)
        if rank != 0 and ok:
            try:
                peer = PeerBuffer(handle=bytes(handle.cpu().numpy().tobytes()))
            except Exception as exc:  # noqa: BLE001
                ok = 0
                print(f"bench.py: rank {rank} could not map rank 0's buffer: {exc}", file=sys.stderr)
        flag = torch.tensor([ok], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if int(flag.item()) == 0:
            if peer is not None:
                peer.close(); peer = None
            collect = "nccl"
    collector = None
    if collect in ("nccl", "local"):
        collector = RingCollector(rank, world, K, (batch, nl), "cuda")
    if peer is not None:
        # every rank's kernels publish "steps done" into rank 0's buffer behind each step (b200pf_series_bind_flag): the agent
        # reads a 4-byte word per rank to know that a step has fully arrived — no collective anywhere in the stepping loop
        eng.series_bind_flag(peer.ptr + ring_bytes + 4 * rank)
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device="cuda")      # > 126 MB L2
    state = {"k": 0}

    def rho_ptr(slot):
        if peer is not None:
            return peer.ptr + 4 * ((rank * 2 * K + slot) * slot_elems)
        return collector.ring[slot].data_ptr()

    def one_step():
        k = state["k"]
        slot = k % (2 * K)
        eng.series_bind_outputs(0, status.data_ptr(), iters.data_ptr(), rho_ptr(slot))
        env.step_device()
        if collector is not None:
            collector.step_done(k)          # (p2p: nothing to launch — results and the completion word are stored by the step's kernels)
        state["k"] = k + 1

    def drain():
        if collector is not None:
            collector.drain()

    n_warm = max(args.warmup, 3)
    for _ in range(n_warm):
        one_step()
    drain()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    launches0 = eng.launch_count + eng.redo_launch_count
    sampler = ClockSampler(local) if rank == 0 else None
    if sampler:
        sampler.start()
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    for a, b in evs:
        flush.zero_()                       # evict L2 between timed iterations (not timed)
        a.record()
        one_step()
        b.record()
    tail_a, tail_b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tail_a.record()
    drain()                                 # outstanding arrival signals / gathers are timed too
    tail_b.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t_wall = time.perf_counter() - t_wall0
    clocks = sampler.stop() if sampler else None
    launches = eng.launch_count + eng.redo_launch_count - launches0
    step_ms = np.array([a.elapsed_time(b) for a, b in evs], dtype=np.float64)
    tail_ms = float(tail_a.elapsed_time(tail_b))
    dev_ms = float(step_ms.sum()) + tail_ms
    n_bad = int((status != 0).sum().item())
    mean_iters = float(iters.float().mean().item())
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    dev_ms_max = float(t.item())
    value = world * batch * args.steps / (dev_ms_max * 1e-3)
    n_series_steps = n_warm + args.steps

    # ---- self-checks of what was just timed -----------------------------------------------------------------------------
    out_h, status_h, iters_h, rho_h = eng.series_fetch()      # rho_h is read back from wherever the kernel stored it (rank 0's HBM)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, gm, out_h, status_h, iters_h, rho_h)
    from grid2op_b200.engine import OutputView
    a_or = OutputView(gm, out_h).a_or
    collected_ok = bool(np.allclose(rho_h, a_or / gm.thermal_limit_a[None, :].astype(np.float32), rtol=1e-6, atol=0, equal_nan=True))
    parity = parity_sample(gm, chron, env, out_h, status_h, n_series_steps) if rank == 0 else None
    if world > 1:
        flag = torch.tensor([1 if collected_ok else 0], dtype=torch.int32, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        collected_ok = bool(int(flag.item()))
    if world > 1:
        # rank 0 compares what sits in ITS memory (slices written by the other ranks' kernels, or gathered by NCCL) with the
        # checksum every rank computes from its own result records
        mine = torch.tensor([float(np.nansum(rho_h.astype(np.float64)))], dtype=torch.float64, device="cuda")
        sums = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(sums, mine)
        if rank == 0:
            last = (state["k"] - 1) % (2 * K)
            if peer is not None:
                flags = peer.read(ring_bytes, world).view(np.int32)
                if not (flags == state["k"]).all():          # every rank's completion word must read "all steps done"
                    collected_ok = False
            for r in range(world):
                if peer is not None:
                    got = peer.read(4 * ((r * 2 * K + last) * slot_elems), slot_elems)
                else:
                    got = collector.gathered(r, state["k"] - 1).cpu().numpy().ravel()
                if not np.isclose(float(np.nansum(got.astype(np.float64))), float(sums[r].item()), rtol=1e-9):
                    collected_ok = False

    # ---- end to end through host buffers (C-ABI staged call), every rank, max over ranks ----------
    eng.set_stream(0)
    collated = env.precollate()                  # one-off data-pipeline step (untimed): step-major pinned copy of the series
    for _ in range(3):
        env.step_host()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rho_max = 0.0
    for _ in range(args.steps):
        out, st = env.step_host()
        rho_max += float((st != 0).sum())          # consume the step's result on the host (done flags; the full
        #                                            observation record `out` sits in pinned host memory)
    e2e_s = time.perf_counter() - t0
    t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_sync = world * batch * args.steps / float(t.item())
    e2e_value, e2e_mode = e2e_sync, "lockstep"
    if args.e2e_groups >= 1:
        # asynchronous vectorised environments: the batch is cut into G groups, each with its own stream; while the host
        # consumes the results of one group (and issues its next step) the others are in flight.  Every instance still
        # gets its results back on the host before its next step is launched; K steps of every instance are timed.
        groups = env.host_groups(args.e2e_groups, direct_out=args.e2e_direct)
        ng = len(groups)
        for g in range(ng):
            env.group_launch(g)
        for _ in range(3):
            for g in range(ng):
                env.group_wait(g); env.group_launch(g)
        for g in range(ng):
            env.group_wait(g)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for g in range(ng):
            env.group_launch(g)
        for k in range(args.steps):
            for g in range(ng):
                out, st = env.group_wait(g)
                rho_max += float((st != 0).sum())
                if k + 1 < args.steps:
                    env.group_launch(g)
        e2e_s = time.perf_counter() - t0
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_value = world * batch * args.steps / float(t.item())
        fl = args.e2e_direct
        e2e_mode = f"{ng} groups in flight" + (", results stored by the kernel straight into pinned host memory" if fl & 1 else "") \
            + (", chronics rows read by the kernel straight from pinned host memory (no copy-engine H2D)" if fl & 2 else "") \
            + (", status/iteration counts stored by the kernel into pinned host memory" if fl & 4 else "")
    h2d, d2h = env.bytes_per_step_host()
    kstats = eng.plan_stats()
    if kstats["last_kernel"].startswith("planned"):
        h2d -= batch * gm.n_topo_in            # the planned kernels work from the cached topology plan: no topology records cross PCIe

    if rank == 0:
        peak, peak_src = measured_peaks()
        surv, comp, b_iter = algorithmic_bytes(gm, mean_iters)
        kern_s = float(np.mean(step_ms)) * 1e-3                  # the event pair of a step brackets its launch(es) only
        achieved = batch * surv / kern_s / 1e9
        info = eng.last_launch_info()
        kernel_tag = f"{kstats['last_kernel']}:{args.workload}:T{info['threads_per_instance']}"
        prof = profiled_traffic(kernel_tag)
        cpu = None
        if world == 1 and not args.no_cpu:
            arm = CpuArm(gm, chron, 8192)
            ts = arm.sample(3, args.cpu_seconds)
            cpu = {"value": float(np.median(8192 / ts)), "unit": UNIT, "cores": arm.nthreads, "kind": "port", "sample": arm.describe(ts),
                   "spread": {"min": float((8192 / ts).min()), "max": float((8192 / ts).max())}}
        rate = world * batch / (step_ms * 1e-3)
        line = {
            "metric": w["metric"], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": n_warm,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": w["scaling"], "vs_baseline": None,
            "dtype": "f64", "data": f"synthetic (bundled {w['env']} chronics rows replayed, DoNothing)",
            "config": {"workload": f"{w['env']} AC Newton-Raphson, batch {batch} envs per GPU, DoNothing rollout",
                       "batch_per_gpu": batch, "global_batch": batch * world, "parallelism": f"dp{world} (independent instances)",
                       "l2": "flushed between timed steps (256 MiB memset, outside the event pair)",
                       "precision": "fp64 state/mismatch/flows, fp32 Jacobian+LU, tol 1e-8 MVA, max_iter 10; pivoting fp64 re-solve of "
                                    "whatever the planned kernel leaves unsolved" + (" (OFF in this run)" if args.no_redo else ""),
                       "launch": info, "kernel": kstats, "kernel_tag": kernel_tag, "mean_newton_iterations": mean_iters, "diverged": n_bad,
                       "result_collection": {"local": "single GPU: rho stays in this GPU's HBM",
                                             "p2p": "kernels store rho AND a per-rank completion word straight into rank 0's HBM (CUDA IPC peer mapping "
                                                    "over NVLink); no collective in the stepping loop (NCCL: set-up and timing reduction only)",
                                             "nccl": f"device ring of 2 x {K} step slots, one asynchronous NCCL gather of a half ring to rank 0 every {K} steps "
                                                     "(overlaps the steps that fill the other half)"}[collect],
                       "collected_equals_results": collected_ok,
                       "wall_s_incl_flush": t_wall},
            "spread": {"unit": UNIT, "min": float(rate.min()), "median": float(np.median(rate)), "max": float(rate.max()),
                       "tail_ms": tail_ms, "what": "per-step CUDA-event times of rank 0, as whole-job rates"},
            "parity_check": parity,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "mode": e2e_mode, "lockstep_value": e2e_sync,
                    "what": "BatchedDoNothing host path (group_launch/group_wait; lockstep_value = step_host()): per step H2D of the chronics rows (from pinned host memory, "
                            + ("pre-collated step-major" if collated else "gathered on the host per step")
                            + "), kernel, D2H of the full result records, host reads the done flags of every instance before "
                              "launching its next step; `value`: the batch is stepped as staggered groups (asynchronous "
                              "vectorised envs), `lockstep_value`: all instances wait for each other every step (2 pipelined chunks).  "
                              "DoNothing only: no action crosses the boundary in the timed region (topology plans are cached)"},
            "gpu_launches": int(launches),
            "clocks": clocks,
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": prof[0] if prof else None, "traffic_source": prof[1] if prof else None, "peak_source": peak_src,
                         "algorithmic_bytes_per_env_step": surv, "b_iter_bytes": b_iter,
                         "compulsory_bytes_per_env_step": comp,
                         "achieved_compulsory_gbs": batch * comp / kern_s / 1e9,
                         "flops_view": flops_view(gm, mean_iters, batch, kern_s, clocks),
                         "note": "fused whole-solve kernel: state never round-trips HBM, the kernel is issue/latency bound (see DESIGN.md)"},
        }
        if cpu is not None:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)
        if parity is not None and not parity["ok"]:
            print(f"bench.py: PARITY CHECK FAILED: {parity}", file=sys.stderr)
            env.close()
            raise SystemExit(3)
        if not collected_ok:
            print("bench.py: collected rho differs from the result records", file=sys.stderr)
            raise SystemExit(4)
    env.close()
    if peer is not None:
        peer.close()
    if world > 1:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--workload", default="case14", choices=sorted(WORKLOADS))
    ap.add_argument("--e2e-direct", type=int, default=6,
                    help="group flags (include/b200pf.h): 1 kernels store results straight into pinned host memory, 2 kernels read "
                         "the chronics rows straight from pinned host memory, 4 status / iteration counts stored straight into pinned host memory")
    ap.add_argument("--e2e-groups", type=int, default=4, help="groups in flight for the end-to-end host path (<=1: lockstep only)")
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="instances per GPU (default: the workload's)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="length of the in-run cpu_baseline sample (N=1)")
    ap.add_argument("--cpu-min-seconds", type=float, default=0.0, help="--impl reference: time more than --steps steps until this long")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-redo", action="store_true", help="measurement only: planned kernel without its pivoting safety net")
    ap.add_argument("--gather-every", type=int, default=64, help="N>1: steps per arrival signal / gather")
    ap.add_argument("--collect", default="nccl", choices=["p2p", "nccl"], help="N>1: how rho reaches rank 0")
    ap.add_argument("--policy", type=int, default=0, choices=[0, 1, 2],
                    help="kernel policy (include/b200pf.h): 0 auto = planned kernel, 1 pivoting kernels only, 2 planned always")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step to DIR/<name>.npy (float32, at most 64 MB; rank 0's instances)")
    args = ap.parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
