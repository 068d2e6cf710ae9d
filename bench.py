"""bench.py -- throughput of the egdst hot path on B200: forward simulation (primary line) and the
backward-induction solve ("solve" object) of BASELINE.json's config[3]
(retirement2 scaled to 10k grid x 100 quadrature nodes x 50 periods + 10M-agent simulation).

    python bench.py --gpus N --steps K --warmup W            # own arm, one rank per GPU (torchrun for N>1)
    python bench.py --impl reference --gpus N --steps K ...   # the reference C (oracle/_ref) on the host cores

A step = one simulation pass of this rank's agents on the device-resident S1 solution: Philox uniforms,
policy-table lookups, full [nsimout, nt, nsim] `sims` output written to HBM plus moments, then (N>1) one
NCCL all-reduce of the moment buffer.  Agents per GPU are fixed (weak scaling).  The solve of S1 does not
shard ("replicas only", DESIGN.md): it is measured on every rank with the same K/W and reported from
rank 0 in the "solve" object with its own roofline, e2e and cpu_baseline.

Only the `cpu_baseline` leg and `--impl reference` execute anything under oracle/ (the unmodified
reference C compiled against the MEX shim), as the thing timed *beside* the product, never inside it.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

SIM_METRIC = "agent-periods/s (sim)"
SOLVE_METRIC = "EGM grid-point-periods/s (solve)"
WORKLOAD = "retirement2-scaled S1: ngridm=10000, ny=100, T=50, interest=0.02, nthrhmax=ngridm; S2 simulation on its solution"
SEED_SHOCKS = 12345
SEED_INIT = 20141


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.isfile(p):
        with open(p) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def committed_traffic(kernel: str, key: str):
    """dram bytes per launch of `kernel` from the committed ncu --set full capture, if it was taken at the same
    launch shape (profiles/traffic.json: {kernel: {key: bytes}}); else None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.isfile(p):
        return None
    try:
        with open(p) as f:
            return json.load(f).get(kernel, {}).get(key)
    except Exception:
        return None


def micro_peaks():
    """Committed on-box ceilings and instruction counts (profiles/micro_peaks.json: tools/micro/peaks.cu + ncu SASS page)."""
    p = os.path.join(ROOT, "profiles", "micro_peaks.json")
    try:
        with open(p) as f:
            return json.load(f)
    except Exception:
        return {}


class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        self.p = None

    def start(self):
        try:
            self.p = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits", "-lms", "20"],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in self.f.read().splitlines():
            parts = [x.strip() for x in line.split(",")]
            if len(parts) < 9:
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for nme, v in zip(names, parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(nme)
        try:
            os.unlink(self.f.name)
        except OSError:
            pass
        if sm:
            out.update(sm_mhz=float(np.median(sm)), sm_max_mhz=float(max(mx)), reasons=sorted(reasons), samples=len(sm))
        return out


def fp64_side(flop_per_launch, launch_ms):
    """The FP64 side of the roofline: flop per launch (2*DFMA+DADD+DMUL thread instructions, counted once with ncu on the
    committed profile) over the live launch duration, against the FP64 FMA rate measured on this pool (tools/micro/peaks.cu)."""
    mp = micro_peaks()
    if not flop_per_launch or not mp.get("fp64_fma_tflops"):
        return None
    ach = flop_per_launch / (launch_ms / 1e3) / 1e12
    return {"achieved_tflops": ach, "peak_tflops_measured": mp["fp64_fma_tflops"], "frac": ach / mp["fp64_fma_tflops"],
            "gather16_l2_Gps_measured": mp.get("gather16_l2_Gps")}


def nominal_units(m) -> int:
    """Solve work units (SURVEY 8d): EGM grid points per solve = periods x feasible (state, decision) pairs x ngridm.
    Every S1 (ist, id) is feasible in every period: 50 x 1 x 2 x 10000 = 1.0e6, identical for both arms."""
    return int(m.nt * m.nst * m.nd * m.ngridm)


def s1_model():
    from egdst_b200 import examples
    return examples.retirement2_scaled()


# =====================================================================================================
# own arm
# =====================================================================================================
def own_arm(a):
    import torch
    import torch.distributed as dist
    from egdst_b200 import capi

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- egdst_b200 has no CPU path (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"  # keep stdout to the one JSON line (NCCL prints its version banner there)
        dist.init_process_group("nccl", device_id=dev)
    hbm_peak, peak_src = measured_peaks()

    m = s1_model()
    m.device = local
    m.compile()
    lib = m._capi()
    stream = torch.cuda.Stream()  # the library launches on this stream; torch events on it time the kernels
    torch.cuda.set_stream(stream)
    lib.set_stream(stream.cuda_stream)
    desc = capi.Desc(m)
    nt, nso = m.nt, m.nsimout()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ------------------------------------------------------------------ solve (replica on every rank)
    sol = lib.solve(m, strict=True)
    stored = sol.units()
    units = nominal_units(m)
    rows = int(sum(x - 1 for x in sol.sizes()[0] if x > 0))
    for _ in range(a.warmup):
        lib.resolve(sol, m)
    barrier()
    l0 = lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        lib.resolve(sol, m)
    e1.record()
    barrier()
    solve_ms = max_over_ranks(e0.elapsed_time(e1) / a.steps)
    solve_launches = lib.launch_count() - l0
    code = sol.status()[0]
    if code:
        raise SystemExit("bench.py: S1 solve reported status %d: %s" % (code, lib.last_error()))
    # per-kernel-class device time (separate, untimed pass; two event records per launch)
    lib.profile_enable(True)
    for _ in range(2):
        lib.resolve(sol, m)
    torch.cuda.synchronize()
    prof = lib.profile_read()
    phases = {k: v for k, v in sol.phase_ms().items() if "." not in k and not k.startswith("-")}  # in-kernel phase timers of the two profiled solves
    lib.profile_enable(False)
    ksum = sum(phases.values()) or 1.0
    egm_launch_ms = phases["egm"] / 2 / max(nt - 1, 1)  # the EGM phase of one period (what used to be one launch)
    # algorithmic bytes of one EGM launch (DESIGN.md): read M,C,V of t+1 (24 B/row), write M,C,V_d per stored point
    egm_bytes = 24.0 * (rows / nt + 1) + 24.0 * (stored / nt)
    solve_alg_bytes = 56.0 * rows  # SURVEY 8(d): 56 B per final grid row per period, whole solve
    # e2e for the solve: the user's call -- egdst_solve (allocation + backward induction) + export of M, D to host
    for _ in range(2):  # steady state of a user loop: the released solution object is re-used (no allocation)
        s2 = lib.solve(m, strict=True)
        s2.export()
        del s2
    t0 = time.perf_counter()
    for _ in range(3):
        s2 = lib.solve(m, strict=True)
        mlen, thlen, Mbuf, Dbuf = s2.export()
        del s2
    solve_e2e_s = (time.perf_counter() - t0) / 3
    solve_obj = {
        "metric": SOLVE_METRIC, "value": units / (solve_ms / 1e3), "unit": "grid-point-periods/s", "ms_per_solve": solve_ms,
        "units_per_solve": units, "stored_points": stored, "final_rows": rows, "interpolation_nodes_per_solve": int((units - units / nt) * m.ny),
        "scaling": "replicas only", "dtype": "f64", "gpu_launches": int(solve_launches),
        "e2e": {"value": units / solve_e2e_s, "unit": "grid-point-periods/s", "ms": solve_e2e_s * 1e3,
                "h2d_bytes_per_step": int(8 * (2 * m.ny + len(m.param) + 2 * m.nnst + m.nst * m.nnst + m.nd * m.nnd)),
                "d2h_bytes_per_step": int(Mbuf.nbytes + Dbuf.nbytes + mlen.nbytes + thlen.nbytes)},
        "roofline": {"bound": "hbm", "kernel": "egdst_k_solve_grid, EGM phase of one period", "achieved": egm_bytes / (egm_launch_ms / 1e3) / 1e9, "peak": hbm_peak,
                     "unit": "GB/s", "frac": egm_bytes / (egm_launch_ms / 1e3) / 1e9 / hbm_peak, "peak_source": peak_src,
                     "traffic": None,  # a phase inside the one solve kernel has no DRAM counter of its own; the whole launch:
                     "whole_kernel_traffic": committed_traffic("egdst_k_solve_grid", "S1"),
                     "algorithmic_bytes_per_launch": egm_bytes, "launch_ms": egm_launch_ms,
                     "whole_solve_GBs": solve_alg_bytes / (solve_ms / 1e3) / 1e9,
                     "fp64": fp64_side(micro_peaks().get("egm_fp64_flop_per_launch_S1"), egm_launch_ms),
                     "note": "FP64-issue/latency-bound, not HBM-bound: ~200 flop per algorithmic byte (SURVEY 8d)"},
        "phase_share": {k: round(v / ksum, 4) for k, v in phases.items() if v},
        "phase_ms_per_solve": {k: round(v / 2, 4) for k, v in phases.items() if v},
        "resends_after_seed": sol.resends(),
    }

    # ------------------------------------------------------------------ simulation (sharded, weak scaling)
    nsim = a.nsim
    free_b, _tot = torch.cuda.mem_get_info()
    need = 8 * nso * nt * nsim
    if need > 0.9 * free_b:
        if a.dump_outputs:  # the dump must come from the same inputs on every run
            raise SystemExit("bench.py: --dump-outputs needs room for all %d agents, but %.1f GB of device memory are free" % (nsim, free_b / 1e9))
        nsim = int(0.9 * free_b / (8 * nso * nt))
    g = torch.Generator(device=dev)
    g.manual_seed(SEED_INIT + rank)
    d_init = torch.empty(2 * nsim, dtype=torch.float64, device=dev)
    d_init[:nsim] = 1.0
    d_init[nsim:] = m.a0 + 0.5 * (m.mmax - m.a0) * torch.rand(nsim, dtype=torch.float64, device=dev, generator=g)
    d_sims = torch.empty(nso * nt * nsim, dtype=torch.float64, device=dev)
    d_mom = torch.zeros(3 * nso * nt, dtype=torch.float64, device=dev)
    agent0 = rank * nsim

    def sim_step(ev=None):
        d_mom.zero_()
        if ev:
            ev[0].record()
        lib.simulate_device(m, sol, d_init.data_ptr(), nsim, agent0, SEED_SHOCKS, d_sims.data_ptr(), d_mom.data_ptr(), desc=desc)
        if ev:
            ev[1].record()
        if world > 1:
            dist.all_reduce(d_mom)

    for _ in range(a.warmup):
        sim_step()
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
    l0 = lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    e0.record()
    for i in range(a.steps):
        sim_step(kev[i])
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    sim_ms = max_over_ranks(e0.elapsed_time(e1) / a.steps)
    if a.dump_outputs and rank == 0:
        dump_sim_outputs(a.dump_outputs, sol, d_sims, d_mom, nsim, nt, nso)
    sim_launches = lib.launch_count() - l0
    kern_ms = float(np.mean([x.elapsed_time(y) for x, y in kev]))
    alive = float(d_mom.view(nt, nso, 3)[:, 0, 2].sum().item())  # agent-periods written (all ranks after the all-reduce)
    sim_units = world * nsim * nt
    if abs(alive - sim_units) > 0.5:
        sim_units = int(alive)  # agents that died or were skipped write no record
    sim_bytes = 8.0 * nso * nt * nsim + 16.0 * nsim  # per launch: sims records out + init in (SURVEY 8d: 8*nsimout B per unit)

    # ------------------------------------------------------------------ strong scaling: BASELINE config[3] as stated,
    # 10M agents IN TOTAL split over the ranks (the primary line above is weak scaling: 10M agents per GPU)
    from egdst_b200.distributed import shard_range
    ns_total = a.strong_nsim
    slo, shi = shard_range(ns_total, rank, world)
    ns = shi - slo
    d_init_s = torch.empty(2 * ns, dtype=torch.float64, device=dev)
    d_init_s[:ns] = 1.0
    d_init_s[ns:] = d_init[nsim:nsim + ns] if ns <= nsim else m.a0 + 0.5 * (m.mmax - m.a0) * torch.rand(ns, dtype=torch.float64, device=dev, generator=g)

    def strong_step():
        d_mom.zero_()
        lib.simulate_device(m, sol, d_init_s.data_ptr(), ns, slo, SEED_SHOCKS, d_sims.data_ptr(), d_mom.data_ptr(), desc=desc)
        if world > 1:
            dist.all_reduce(d_mom)

    for _ in range(a.warmup):
        strong_step()
    barrier()
    s0, s1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s0.record()
    for _ in range(a.steps):
        strong_step()
    s1.record()
    barrier()
    strong_ms = max_over_ranks(s0.elapsed_time(s1) / a.steps)
    strong = {"metric": SIM_METRIC, "value": ns_total * nt / (strong_ms / 1e3), "unit": "agent-periods/s", "ms_per_step": strong_ms, "scaling": "strong",
              "config": {"workload": "S2 as BASELINE config[3] states it: %d agents in total, sharded over %d GPU(s), moments all-reduced" % (ns_total, world),
                         "agents_per_gpu": ns}}

    # e2e: the host-buffer C-ABI call a MEX gateway makes -- init from pinned host memory, full sims array back to host
    ne = min(a.e2e_nsim, nsim)
    h_init = torch.empty(2 * ne, dtype=torch.float64).pin_memory()
    h_init[:ne] = 1.0
    h_init[ne:] = m.a0 + 0.5 * (m.mmax - m.a0) * torch.rand(ne, dtype=torch.float64)
    h_sims = torch.empty(nso * nt * ne, dtype=torch.float64).pin_memory()
    dp = C.POINTER(C.c_double)

    def e2e_step():
        rc = lib.L.egdst_simulate_philox(C.byref(desc.c), sol.handle, 0, C.cast(h_init.data_ptr(), dp), ne, agent0, SEED_SHOCKS,
                                         C.cast(h_sims.data_ptr(), dp), None)
        if rc:
            raise SystemExit("bench.py: e2e simulate failed: " + lib.last_error())

    e2e_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.e2e_steps):
        e2e_step()
    torch.cuda.synchronize()
    e2e_s = max_over_ranks((time.perf_counter() - t0) / a.e2e_steps)
    e2e = {"value": world * ne * nt / e2e_s, "unit": "agent-periods/s", "h2d_bytes_per_step": int(16 * ne),
           "d2h_bytes_per_step": int(8 * nso * nt * ne), "agents_per_gpu": ne, "ms": e2e_s * 1e3,
           "api": "egdst_simulate_philox (host init in, host sims out; pinned buffers)",
           "sample": "1/%d of the headline workload: %d of %d agents per GPU (the leg is bound by the device-to-host copy of the path array, so its rate does not depend on the agent count)" % (max(nsim // max(ne, 1), 1), ne, nsim),
           "d2h_GBs_aggregate": world * 8.0 * nso * nt * ne / e2e_s / 1e9,
           "limiter": "device-to-host copy of the [nsimout, nt, nsim] path array (PCIe / host memory): all GPUs of the box drain into the same host"}

    # the moments-only entry point (no path array crosses PCIe): what an estimation loop calls
    h_mom = torch.zeros(3 * nso * nt, dtype=torch.float64).pin_memory()
    nm_agents = min(nsim, 10_000_000)
    h_init_m = torch.empty(2 * nm_agents, dtype=torch.float64).pin_memory()
    h_init_m[:nm_agents] = 1.0
    h_init_m[nm_agents:] = m.a0 + 0.5 * (m.mmax - m.a0) * torch.rand(nm_agents, dtype=torch.float64)

    def e2e_mom_step():
        rc = lib.L.egdst_simulate_philox(C.byref(desc.c), sol.handle, 0, C.cast(h_init_m.data_ptr(), dp), nm_agents, agent0, SEED_SHOCKS,
                                         None, C.cast(h_mom.data_ptr(), dp))
        if rc:
            raise SystemExit("bench.py: e2e moments failed: " + lib.last_error())

    e2e_mom_step()
    barrier()
    t0 = time.perf_counter()
    for _ in range(a.e2e_steps):
        e2e_mom_step()
    torch.cuda.synchronize()
    e2e_mom_s = max_over_ranks((time.perf_counter() - t0) / a.e2e_steps)
    e2e["moments_only"] = {"value": world * nm_agents * nt / e2e_mom_s, "unit": "agent-periods/s", "agents_per_gpu": nm_agents, "ms": e2e_mom_s * 1e3,
                           "h2d_bytes_per_step": int(16 * nm_agents), "d2h_bytes_per_step": int(8 * 3 * nso * nt),
                           "api": "egdst_simulate_philox(sims=NULL, moments): host init in, [3,nsimout,nt] moments out"}

    # ------------------------------------------------------------------ BASELINE config[4]: the batched estimation sweep
    batch = None
    if not a.no_batch:
        lib.set_stream(stream.cuda_stream)
        batch = measure_batch(a, rank, world, dev, with_cpu=(world == 1 and not a.no_cpu))

    # cpu baseline: the unmodified reference C on one host core (it is single-threaded), rank 0 at N=1 only
    cpu = None
    if rank == 0 and world == 1 and not a.no_cpu:
        cpu, solve_cpu = cpu_baseline(m, sol, a)
        solve_obj["cpu_baseline"] = solve_cpu

    if rank == 0:
        line = {
            "metric": SIM_METRIC, "value": sim_units / (sim_ms / 1e3), "unit": "agent-periods/s", "n_gpus": world, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": sim_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f64", "data": "synthetic",
            "config": {"workload": WORKLOAD, "agents_per_gpu": nsim, "agents_total": world * nsim, "periods": nt, "nsimout": nso,
                       "output": "full sims [nsimout, nt, nsim] + moments", "rng": "Philox4x32-10, counter=(global agent id, period)",
                       "parallelism": "agents sharded, dp%d" % world, "l2": "outputs (%.1f GB per step) larger than L2" % (sim_bytes / 1e9)},
            "gpu_launches": int(sim_launches),
            "clocks": clocks,
            "e2e": e2e,
            "roofline": {"bound": "hbm", "kernel": "egdst_k_simulate", "achieved": sim_bytes / (kern_ms / 1e3) / 1e9, "peak": hbm_peak, "unit": "GB/s",
                         "frac": sim_bytes / (kern_ms / 1e3) / 1e9 / hbm_peak, "peak_source": peak_src,
                         "traffic": committed_traffic("egdst_k_simulate", "nsim=%d" % nsim),
                         "algorithmic_bytes_per_launch": sim_bytes, "launch_ms": kern_ms,
                         "fp64": fp64_side((micro_peaks().get("sim_fp64_flop_per_launch_nsim10M") or 0) * nsim / 1e7 or None, kern_ms)},
            "cpu_baseline": cpu,
            "solve": solve_obj,
            "strong": strong,
            "batch": batch,
        }
        emit(line)
    if world > 1:
        dist.destroy_process_group()


# =====================================================================================================
# BASELINE config[4], the batched estimation sweep (S3): part of the default line ("batch" object) and a workload of its own
# =====================================================================================================
def measure_batch(a, rank, world, dev, with_cpu):
    """4096 deaton2 parameter vectors, block-partitioned over the ranks (strong scaling): one batched solve, one
    batched moments-only simulation of 1024 agents under every vector, one all-reduce that assembles the moment
    table [nvec, 3, nsimout, nt] on every rank.  A step = the whole sweep.  Returns the result object on rank 0."""
    import torch
    import torch.distributed as dist
    from egdst_b200 import capi, examples
    from egdst_b200.distributed import shard_range
    m = examples.deaton2(); m.device = dev.index; m.compile()
    lib = m._capi()
    lib.set_stream(torch.cuda.current_stream().cuda_stream)
    nvec, nsim = a.batch_nvec, a.batch_nsim
    rng = np.random.default_rng(4096)
    params = np.column_stack([rng.uniform(0.0, 0.05, nvec), rng.uniform(0.75, 1.75, nvec)])
    lo, hi = shard_range(nvec, rank, world)
    mine = np.ascontiguousarray(params[lo:hi])
    sol = lib.solve_batch(m, mine)
    nso, nt = m.nsimout(), m.nt
    nmom = 3 * nso * nt
    d_init = torch.empty(2 * nsim, dtype=torch.float64, device=dev); d_init[:nsim] = 1.0; d_init[nsim:] = 0.25
    table = torch.zeros(nvec * nmom, dtype=torch.float64, device=dev)
    desc = capi.Desc(m)

    def step():
        lib.resolve(sol, m, mine)
        table.zero_()
        lib.sim_moments_device(m, sol, d_init.data_ptr(), nsim, 0, 7, table.data_ptr() + 8 * lo * nmom, desc=desc)
        if world > 1:
            dist.all_reduce(table)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(a.warmup):
        step()
    barrier()
    l0 = lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(a.steps):
        step()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1) / a.steps
    if a.dump_outputs and rank == 0:  # a fixed sample of 1024 of the sweep's vectors keeps the dump small
        vecs = np.sort(np.random.default_rng(4096).choice(nvec, min(nvec, 1024), replace=False))
        _save(a.dump_outputs, "batch_vectors", vecs)
        _save(a.dump_outputs, "batch_moments", table.view(nvec, nt, nso, 3)[torch.from_numpy(vecs).to(dev)].permute(0, 3, 2, 1).cpu().numpy())
    if world > 1:
        t = torch.tensor([ms], dtype=torch.float64, device=dev); dist.all_reduce(t, op=dist.ReduceOp.MAX); ms = float(t.item())
    # split of one step on this rank (events around the two calls, outside the timed region)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    ev[0].record(); lib.resolve(sol, m, mine); ev[1].record()
    lib.sim_moments_device(m, sol, d_init.data_ptr(), nsim, 0, 7, table.data_ptr() + 8 * lo * nmom, desc=desc); ev[2].record()
    torch.cuda.synchronize()
    bad = sum(1 for v in range(hi - lo) if sol.status(v)[0])
    if rank != 0:
        return None
    units = nvec * nominal_units(m)
    out = {"metric": "parameter vectors/s (batched solve + simulated moments)", "value": nvec / (ms / 1e3), "unit": "vectors/s", "n_gpus": world,
           "steps": a.steps, "warmup": a.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "dtype": "f64", "data": "synthetic",
           "config": {"workload": "S3: %d deaton2 parameter vectors (interest~U[0,.05], income~U[.75,1.75], default_rng(4096)), %d agents each, moments all-reduced" % (nvec, nsim),
                      "parallelism": "parameter vectors sharded, dp%d" % world},
           "gpu_launches": int(lib.launch_count() - l0), "solve_units_per_s": units / (ms / 1e3), "agent_periods_per_s": nvec * nsim * nt / (ms / 1e3),
           "ms_solve_rank0": ev[0].elapsed_time(ev[1]), "ms_moments_rank0": ev[1].elapsed_time(ev[2]),
           "vectors_with_error_status_on_rank0": bad}
    if with_cpu:
        out["cpu_baseline"] = batch_cpu_baseline(params, nsim, a)
    return out


def dump_sim_outputs(out, sol, d_sims, d_mom, nsim, nt, nso):
    """What the timed path returned in its last step: the S1 solution (cells stacked in (it, ist) order, with their row
    counts), the moments [3, nsimout, nt] and the records [k, nt, nsimout] of a fixed sample of k = 1024 agents (the full
    path array is tens of GB)."""
    import torch
    M, D = sol.M, sol.D
    cells = [(M[ist][it], D[ist][it]) for it in range(nt) for ist in range(len(M)) if M[ist][it] is not None and M[ist][it].size]
    _save(out, "solve_M", np.concatenate([c[0] for c in cells]))
    _save(out, "solve_D", np.concatenate([c[1] for c in cells]))
    _save(out, "solve_cell_rows", np.array([[c[0].shape[0], c[1].shape[0]] for c in cells], dtype=np.float64))
    _save(out, "sim_moments", d_mom.view(nt, nso, 3).permute(2, 1, 0).cpu().numpy())
    k = min(nsim, 1024)
    agents = np.sort(np.random.default_rng(SEED_SHOCKS).choice(nsim, k, replace=False))
    _save(out, "sim_agents", agents.astype(np.float64))
    _save(out, "sim_records", d_sims.view(nsim, nt, nso)[torch.from_numpy(agents).to(d_sims.device)].cpu().numpy())


DUMP_CAP = 64 * 2 ** 20
_dumped = [0]


def _save(out, name, arr):
    """DIR/<name>.npy with every entry finite, and DIR/<name>_nonfinite.npy coding the entries that were not (0 finite,
    1 NaN, 2 +inf, 3 -inf; they are 0 in <name>.npy).  -inf is a value the solver and simulator do return (consumption
    and value at zero consumption, and the moments summing them); NaN marks simulation columns a model leaves unset.
    Split this way, two dumps compare entry by entry with a tolerance and still agree on every non-finite value."""
    os.makedirs(out, exist_ok=True)
    a = np.asarray(arr, dtype=np.float64)
    code = np.zeros(a.shape, dtype=np.float32)
    code[np.isnan(a)] = 1
    code[a == np.inf] = 2
    code[a == -np.inf] = 3
    _dumped[0] += a.nbytes + code.nbytes
    if _dumped[0] > DUMP_CAP:
        raise SystemExit("bench.py: --dump-outputs would exceed %d MB at %s" % (DUMP_CAP >> 20, name))
    np.save(os.path.join(out, name + ".npy"), np.where(code == 0, a, 0.0))
    np.save(os.path.join(out, name + "_nonfinite.npy"), code)


def _batch_worker(job):
    from egdst_b200 import examples
    from tests.oracles import oracle_for
    interest, income, nsim, seed = job
    mi = examples.deaton2(interest=float(interest), income=float(income))
    o = oracle_for(mi)
    Mr, Dr = o.solve()
    s = o.seconds
    init = np.column_stack([np.ones(nsim), np.full(nsim, 0.25)])
    rs = np.random.default_rng(seed).random(4 * nsim * mi.nt)
    o.simulate(Mr, Dr, init, rs, 0)
    return s + o.seconds


def batch_cpu_baseline(params, nsim, a):
    """The reference C on every host core (BASELINE.md section 4): `cores` independent single-threaded reference
    processes, each solving and simulating its share of a bounded sample of the sweep's vectors.  None where the
    reference is not built (oracle/ref.py)."""
    import multiprocessing as mp
    from egdst_b200 import examples
    from tests.oracles import ref_available
    if not ref_available(examples.deaton2()):
        return None
    cores = os.cpu_count() or 1
    nv = max(cores, min(a.batch_cpu_nvec, params.shape[0]))
    jobs = [(params[i, 0], params[i, 1], nsim, i) for i in range(nv)]
    ctx = mp.get_context("fork")
    t0 = time.perf_counter()
    with ctx.Pool(cores) as pool:
        gate = pool.map(_batch_worker, jobs)
    wall = time.perf_counter() - t0
    return {"value": nv / wall, "unit": "vectors/s", "cores": cores, "kind": "reference",
            "sample": "%d of the sweep's vectors, solved and simulated (%d agents) by %d reference processes; wall %.2f s, gateway time per vector %.2f ms" % (nv, nsim, cores, wall, 1e3 * float(np.mean(gate)))}


def batch_arm(a):
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("", "VERSION"):
            os.environ["NCCL_DEBUG"] = "WARN"
        dist.init_process_group("nccl", device_id=dev)
    stream = torch.cuda.Stream(); torch.cuda.set_stream(stream)
    out = measure_batch(a, rank, world, dev, with_cpu=(world == 1 and not a.no_cpu))
    if rank == 0:
        out["vs_baseline"] = None
        emit(out)
    if world > 1:
        dist.destroy_process_group()


def cpu_baseline(m, sol, a):
    """Reference C (oracle/_ref) on one core: simulate a bounded sample of agents on the exported tables, and one S1 solve.
    Where the reference is not built, the simulation is timed with its C restatement (oracle/port) and the solve is
    not timed (the solver has no restatement)."""
    from tests.oracles import oracle_for
    orc = oracle_for(m)
    kind = orc.kind if orc.kind == "reference" else "port"
    M, D = sol.M, sol.D
    ns = a.cpu_nsim
    rng = np.random.default_rng(SEED_INIT)
    init = np.column_stack([np.ones(ns), m.a0 + 0.5 * (m.mmax - m.a0) * rng.random(ns)])
    rs = rng.random(4 * ns * m.nt)
    orc.simulate(M, D, init, rs, 0)
    sim_s = orc.seconds
    cpu = {"value": ns * m.nt / sim_s, "unit": "agent-periods/s", "cores": 1, "kind": kind,
           "sample": "%d agents x %d periods on the S1 tables, gateway time %.2f s (reference simulator is single-threaded)" % (ns, m.nt, sim_s),
           "host_cores": os.cpu_count()}
    solve_cpu = None
    if not a.no_cpu_solve and kind == "reference":
        orc.solve()
        s = orc.seconds
        solve_cpu = {"value": nominal_units(m) / s, "unit": "grid-point-periods/s", "cores": 1, "kind": orc.kind,
                     "sample": "one full S1 solve, gateway time %.2f s (reference solver is single-threaded)" % s, "host_cores": os.cpu_count()}
    return cpu, solve_cpu


# =====================================================================================================
# reference arm: the unmodified reference C on the host cores
# =====================================================================================================
_W = {}


def _worker_init(M, D):
    from tests.oracles import oracle_for
    m = s1_model()
    _W["m"], _W["orc"], _W["M"], _W["D"] = m, oracle_for(m), M, D


def _worker_sim(job):
    seed, ns = job
    m, orc = _W["m"], _W["orc"]
    rng = np.random.default_rng(seed)
    init = np.column_stack([np.ones(ns), m.a0 + 0.5 * (m.mmax - m.a0) * rng.random(ns)])
    rs = rng.random(4 * ns * m.nt)
    orc.simulate(_W["M"], _W["D"], init, rs, 0)
    return orc.seconds  # clock_gettime around the reference's mexFunction only (BASELINE.md section 4)


def reference_arm(a):
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if rank != 0:
        return
    import multiprocessing as mp
    from tests.oracles import oracle_for
    m = s1_model()
    orc = oracle_for(m)
    t0 = time.perf_counter()
    M, D = orc.solve()
    solve_s = orc.seconds
    units = nominal_units(m)
    cores = os.cpu_count() or 1
    per = max(a.ref_nsim // cores, 1)
    ctx = mp.get_context("fork")
    with ctx.Pool(cores, initializer=_worker_init, initargs=(M, D)) as pool:
        def step(i):
            # the step ends when the slowest of the concurrent gateways ends
            return max(pool.map(_worker_sim, [(1000 * i + k, per) for k in range(cores)]))
        for i in range(a.warmup):
            step(i)
        t = [step(100 + i) for i in range(a.steps)]
    sec = float(np.mean(t))
    val = cores * per * m.nt / sec
    sample = "%d agents x %d periods per step, split over %d independent single-threaded reference processes" % (cores * per, m.nt, cores)
    line = {
        "impl": "reference", "metric": SIM_METRIC, "value": val, "unit": "agent-periods/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": WORKLOAD, "sample": sample},
        "gpu_launches": 0,
        "cpu_baseline": {"value": val, "unit": "agent-periods/s", "cores": cores, "kind": orc.kind, "sample": sample},
        "e2e": {"value": val, "unit": "agent-periods/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "solve": {"metric": SOLVE_METRIC, "value": units / solve_s, "unit": "grid-point-periods/s", "ms_per_solve": solve_s * 1e3,
                  "cores": 1, "kind": orc.kind, "sample": "one full S1 solve (the reference solver is single-threaded)", "units_per_solve": units},
    }
    emit(line)


_JSON_FD = None


def _guard_stdout():
    """Keep the process's stdout for the one JSON line: everything else that writes to file descriptor 1 -- NCCL
    prints its version banner there whenever NCCL_DEBUG is set, whatever the level -- goes to stderr."""
    global _JSON_FD
    if _JSON_FD is None:
        sys.stdout.flush()
        _JSON_FD = os.dup(1)
        os.dup2(2, 1)


def emit(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _JSON_FD is None:
        sys.stdout.write(data.decode()); sys.stdout.flush()
    else:
        os.write(_JSON_FD, data)


def main():
    _guard_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--nsim", type=int, default=int(os.environ.get("EGDST_BENCH_NSIM", 10_000_000)), help="agents per GPU")
    ap.add_argument("--e2e-nsim", type=int, default=1_000_000)
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--cpu-nsim", type=int, default=700_000, help="agents of the CPU baseline sample (about 11 s of the reference simulator on one core)")
    ap.add_argument("--ref-nsim", type=int, default=400_000)
    ap.add_argument("--workload", default="s1s2", choices=["s1s2", "batch"], help="s1s2: BASELINE config[3] (default); batch: config[4] sweep")
    ap.add_argument("--batch-nvec", type=int, default=4096)
    ap.add_argument("--batch-nsim", type=int, default=1024)
    ap.add_argument("--batch-cpu-nvec", type=int, default=4096, help="vectors of the sweep the CPU baseline solves and simulates (all host cores)")
    ap.add_argument("--strong-nsim", type=int, default=10_000_000, help="agents IN TOTAL of the strong-scaling object")
    ap.add_argument("--no-batch", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-cpu-solve", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the timed paths computed in their last step to DIR/<name>.npy (non-finite entries coded in DIR/<name>_nonfinite.npy; at most 64 MB; e.g. dumps/)")
    a = ap.parse_args()
    a.warmup = max(a.warmup, 3) if a.impl == "own" else a.warmup
    if a.impl == "reference":
        reference_arm(a)
    elif a.workload == "batch":
        batch_arm(a)
    else:
        own_arm(a)


if __name__ == "__main__":
    main()
