#!/usr/bin/env python
"""bench.py -- BASELINE.json's metric: FR3 RNEA+FD evals/sec (fp64) on N B200s, with roofline fractions.

    python bench.py --gpus 1 --steps 10 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...     # the reference arm: the CPU oracle on all host threads
    python bench.py ... --dump-outputs DIR   # also write the last timed step's tau and qdd (a fixed sample) to DIR

One step = one batched RNEA pass (BASELINE.json configs[1]) + one batched forward-dynamics pass (configs[2]) over
2^24 synthetic FR3 states per GPU, device-resident SoA, sampled on the device by the counter-based generator of
SURVEY.md 8d.  Each GPU owns its own 2^24 states (weak scaling, no data-path collective).  Prints ONE JSON line.

The same line carries, under `configs`, short legs of the other BASELINE.json configurations so that every run the
driver makes (1, 2, 4, 8 GPUs) records them: `fused_rnea_fd` (the one-pass kernel behind multibody_rnea_fd_batch),
`rollout` (configs[3]: 65 536 trajectories x 64 steps split over the ranks, strong scaling) and `chain32` (configs[4]:
2^26 states of the 32-joint chain split over the ranks, strong scaling), each with its own roofline object.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "FR3 RNEA+FD evals/sec (fp64)"
UNIT = "evals/s"
STATES_PER_GPU = 1 << 24
# algorithmic work per evaluation (SURVEY.md 8d / BASELINE.md section 2), N = 7
RNEA_FLOPS, FD_FLOPS, BYTES_PER_EVAL = 2026.0, 4180.0, 224.0
SEED_RNEA, SEED_FD = 0x5EED0001, 0x5EED0002
# FP64-pipe SASS instructions of the fr3-specialised kernels (tools/sass_count.sh; tests/test_host.py checks the static
# totals against the built library).  The kernels are straight-line except for the out-of-range fallback of the batched
# sin/cos (rb_sincos_batched: six per-joint CUDA sincos() calls, 21 FP64 instructions each, taken only when some
# |q_i| >= 1e5): executed per state = static - fallback.  ncu's smsp__sass_thread_inst_executed_op_d{fma,add,mul}
# counters in profiles/ agree.
FP64_STATIC = {"rb_rnea_kernel": 804, "rb_fd_kernel": 1299}
FP64_FALLBACK = {"rb_rnea_kernel": 126, "rb_fd_kernel": 126}
FP64_INSTR = {k: FP64_STATIC[k] - FP64_FALLBACK[k] for k in FP64_STATIC}
FP64_LANES_PER_SM = 64
# --dump-outputs: states written per array, chosen once by a fixed seed so that two builds compare output for output
DUMP_STATES, DUMP_SEED = 1 << 18, 0x5EED00D0


def profiled(kernel):
    """What the committed `ncu --set full` capture of `kernel` says about ONE launch: DRAM bytes moved and (captures of
    round 2 on) executed FP64 instructions by opcode.  The last match wins: the capture named *final* if there is one."""
    best = None
    pdir = os.path.join(ROOT, "profiles")
    names = sorted(os.listdir(pdir), key=lambda nm: ("final" in nm, nm)) if os.path.isdir(pdir) else []

    def num(v):
        x, unit = (v.split() + [""])[:2]
        return float(x) * {"Gbyte": 1e9, "Mbyte": 1e6, "Kbyte": 1e3, "byte": 1.0, "inst": 1.0, "": 1.0}.get(unit, 1.0)

    for name in names:
        if not name.endswith("ncu_full_summary.json"):
            continue
        with open(os.path.join(pdir, name)) as f:
            for row in json.load(f):
                if kernel in row.get("kernel", "") and "dram__bytes_read.sum" in row:
                    d = {"bytes": num(row["dram__bytes_read.sum"]) + num(row["dram__bytes_write.sum"]), "source": "profiles/" + name,
                         "grid": num(row.get("launch__grid_size", "0")), "block": num(row.get("launch__block_size", "0"))}
                    ops = [row.get(f"smsp__sass_thread_inst_executed_op_{o}_pred_on.sum") for o in ("dfma", "dadd", "dmul")]
                    if all(ops):
                        d["fp64_thread_flops"] = 2 * num(ops[0]) + num(ops[1]) + num(ops[2])
                        # every instruction the FP64 pipe executed (DSETP and conversions included), per thread
                        pipe = row.get("sm__inst_executed_pipe_fp64.sum")
                        d["fp64_thread_instr"] = 32.0 * num(pipe) if pipe else sum(num(o) for o in ops)
                    best = d
    return best


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler(threading.Thread):
    """Samples SM clock, power and throttle reasons of one GPU DURING the timed region (B200_PROFILING.md recipe).
    NVML through pynvml (a query takes ~0.1 ms, so even a 20 ms timed region gets several samples); falls back to
    polling nvidia-smi when pynvml is unavailable."""
    REASONS = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self._stop_evt = index, [], threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and all(x.strip().isdigit() for x in visible.split(",")) else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM))
            self._reasons = getattr(pynvml, "nvmlDeviceGetCurrentClocksEventReasons", None) or pynvml.nvmlDeviceGetCurrentClocksThrottleReasons
            self.nvml = pynvml
        except Exception:
            self.nvml = None

    def run(self):
        if self.nvml is not None:
            nv = self.nvml
            while not self._stop_evt.is_set():
                try:
                    self.rows.append((float(nv.nvmlDeviceGetClockInfo(self.handle, nv.NVML_CLOCK_SM)),
                                      nv.nvmlDeviceGetPowerUsage(self.handle) / 1000.0,
                                      int(self._reasons(self.handle))))
                except Exception:
                    pass
                self._stop_evt.wait(0.002)
            return
        fields = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
                  "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self._stop_evt.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={fields}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout
                p = [x.strip() for x in out.strip().split(",")]
                if len(p) == 7:
                    mask = sum(bit for bit, k in zip((0x8, 0x40, 0x20, 0x4), range(3, 7)) if p[k].lower().startswith("active"))
                    self.max_mhz = float(p[1])
                    self.rows.append((float(p[0]), float(p[2]), mask))
            except Exception:
                pass
            self._stop_evt.wait(0.1)

    def stop(self):
        self._stop_evt.set()
        self.join(timeout=6)
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm = sorted(r[0] for r in self.rows)
        mask = 0
        for r in self.rows:
            mask |= r[2]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": getattr(self, "max_mhz", None),
                "reasons": [name for bit, name in self.REASONS.items() if mask & bit],
                "power_w_max": max(r[1] for r in self.rows), "samples": len(self.rows),
                "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ----------------------------------------------------------------------------- CPU arm (oracle; test infrastructure)
def host_threads():
    # torchrun exports OMP_NUM_THREADS=1: size the team from the CPUs this process may run on instead
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


def cpu_single_state(orc, calls=1_000_000):
    """BASELINE.json configs[0]: the single-state RNEA of the reference path on ONE host core, at the reference's two
    inputs -- q = dq = ddq = 0 (`bench_rnea`, multibody.rs:204-209) and the state of rigidbody_bindings/main.cpp:103-105 --
    `calls` evaluations each after a 10 % warm-up (one C loop over a batch of identical states: no Python per call)."""
    states = {"zero_state": (np.zeros(7), np.zeros(7), np.zeros(7)),
              "main_cpp_state": (np.array([0, 0, 1, 0, 1, 0, 0.0]), np.array([0, 0, 0, 0, 1, 0, 0.0]), np.array([1, 0, 0, 0, 0, 1, 0.0]))}
    out = {"calls": calls}
    for name, (q, dq, ddq) in states.items():
        Q, DQ, DDQ = (np.ascontiguousarray(np.repeat(x[:, None], calls, 1)) for x in (q, dq, ddq))
        orc.rnea_batch(Q[:, : calls // 10], DQ[:, : calls // 10], DDQ[:, : calls // 10], threads=1)
        t0 = time.perf_counter()
        orc.rnea_batch(Q, DQ, DDQ, threads=1)
        out[name + "_ns"] = (time.perf_counter() - t0) / calls * 1e9
    return out


def cpu_arm(sample_states, steps, warmup, single_calls=1_000_000):
    """Times oracle/rb_oracle.c (reference-shaped C restatement; the Rust crate cannot be built in this image),
    OpenMP static chunks over all host threads: RNEA + FD over `sample_states` states per step."""
    from oracle.rb_oracle import Oracle
    orc = Oracle.from_urdf(os.path.join(ROOT, "assets", "fr3.urdf"), fast=True)   # rebuilt -march=native on this host
    m = orc.model
    threads = host_threads()
    if sample_states is None:       # calibrate to ~4 s of wall time per step
        S0 = 1 << 14
        q = orc.fill(SEED_RNEA, 0, m.lower, m.upper, 0, S0); dq = orc.fill(SEED_RNEA, 1, -m.velocity, m.velocity, 0, S0)
        t0 = time.perf_counter()
        orc.rnea_batch(q, dq, q, threads=threads); orc.forward_dynamics_batch(q, dq, q, threads=threads)
        per = (time.perf_counter() - t0) / S0
        sample_states = int(min(1 << 22, max(1 << 14, 4.0 / per)))
    S = sample_states
    q = orc.fill(SEED_RNEA, 0, m.lower, m.upper, 0, S)
    dq = orc.fill(SEED_RNEA, 1, -m.velocity, m.velocity, 0, S)
    ddq = orc.fill(SEED_RNEA, 2, -10.0, 10.0, 0, S)
    tau = orc.fill(SEED_FD, 3, -m.effort, m.effort, 0, S)
    times = []
    for it in range(warmup + steps):
        t0 = time.perf_counter()
        orc.rnea_batch(q, dq, ddq, threads=threads)
        orc.forward_dynamics_batch(q, dq, tau, threads=threads)
        if it >= warmup:
            times.append(time.perf_counter() - t0)
    sec = sum(times) / len(times)
    single = cpu_single_state(orc, single_calls)
    return {"value": 2.0 * S / sec, "unit": UNIT, "cores": threads, "kind": "port",
            "single_state_rnea_ns_one_core": single["zero_state_ns"], "single_state": single,
            "sample": f"{S} FR3 states per step (RNEA + FD each), {steps} timed steps, OpenMP static over {threads} threads, "
                      f"oracle/rb_oracle.c -O3 -march=native"}, sec, S


def run_reference(args, rank):
    if rank != 0:
        return
    cb, sec, S = cpu_arm(None, max(1, args.steps), max(1, args.warmup))
    line = {"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": "fr3_rnea+fd", "states_per_step": S, "layout": "soa",
                       "note": "CPU port of the reference path (oracle/); the Rust crate cannot be built here (no cargo; probed)"},
            "cpu_baseline": cb,
            "e2e": {"value": cb["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------- GPU arm
def bare_copy_ms(up_bytes, down_bytes, reps, dev, barrier):
    """Milliseconds one rank needs to move `up_bytes` host -> device and `down_bytes` device -> host at the same time with
    plain pinned copies (no kernel): the ceiling of the end-to-end figure.  Collective: every rank calls it; allocation and
    a warm-up pass come first, then a barrier, then the timed passes -- so the ranks really compete for the host's memory."""
    import torch
    cap, piece = 2 << 30, 64 << 20
    nu, nd = max(1, min(cap, up_bytes)), max(1, min(cap, down_bytes))
    hu = torch.empty(nu, dtype=torch.uint8, pin_memory=True); du = torch.empty(nu, dtype=torch.uint8, device=dev)
    hd = torch.empty(nd, dtype=torch.uint8, pin_memory=True); dd = torch.zeros(nd, dtype=torch.uint8, device=dev)
    hu.fill_(1)
    s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def one_pass():
        with torch.cuda.stream(s_up):
            for off in range(0, up_bytes, piece):
                ho = off % nu; ln = min(piece, up_bytes - off, nu - ho)
                du[ho:ho + ln].copy_(hu[ho:ho + ln], non_blocking=True)
        with torch.cuda.stream(s_dn):
            for off in range(0, down_bytes, piece):
                ho = off % nd; ln = min(piece, down_bytes - off, nd - ho)
                hd[ho:ho + ln].copy_(dd[ho:ho + ln], non_blocking=True)
        s_up.synchronize(); s_dn.synchronize()

    one_pass()
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    for _ in range(reps):
        one_pass()
    ms = (time.perf_counter() - t0) * 1e3 / reps
    barrier()
    del hu, hd, du, dd
    return ms


def fp64_roofline(kernel, ms, units, instr_per_unit, flops_executed_per_unit, alg_flops_per_unit, bytes_per_unit,
                  fp64_peak, peak_note, hbm_peak, hbm_src, traffic=None, traffic_src=None, instr_src="static SASS count"):
    """The roofline object of one FP64-pipe-bound kernel.  `frac` is the share of the FP64 pipe's issue slots the launch
    used: every FP64 instruction (DFMA, DADD, DMUL, DSETP...) occupies the pipe like a DFMA, so executed instructions x 2
    (FMA-equivalent flops) per second over the DFMA rate measured on this GPU in this run.  The SURVEY 8d flop count of
    the general algorithm is kept as `algorithmic_frac` (> the executed figure where compile-time constants delete
    work) and the HBM side sits beside it."""
    sec = ms * 1e-3
    fma_eq = 2.0 * instr_per_unit * units / sec / 1e12
    d = {"kernel": kernel, "bound": "fp64", "achieved": fma_eq, "peak": fp64_peak, "unit": "TFLOP/s (FMA-equivalent: 2 x FP64 instructions executed)",
         "frac": fma_eq / fp64_peak, "frac_of_nominal_peak": fma_eq / 37.2, "traffic": traffic, "traffic_source": traffic_src,
         "fp64_instr_per_unit": instr_per_unit, "fp64_instr_source": instr_src,
         "executed_tflops": flops_executed_per_unit * units / sec / 1e12 if flops_executed_per_unit else None,
         "algorithmic_flops_per_unit": alg_flops_per_unit, "algorithmic_tflops": alg_flops_per_unit * units / sec / 1e12,
         "algorithmic_frac": alg_flops_per_unit * units / sec / 1e12 / fp64_peak,
         "units_per_s": units / sec, "ms": ms, "peak_source": peak_note}
    if bytes_per_unit:
        gbs = bytes_per_unit * units / sec / 1e9
        d["hbm"] = {"achieved": gbs, "peak": hbm_peak, "unit": "GB/s", "frac": gbs / hbm_peak, "bytes_per_unit": bytes_per_unit,
                    "peak_source": hbm_src}
    return d


def dump_outputs(out_dir, arrays):
    """Writes each [n, B] float64 device array as out_dir/<name>.npy.  Where B > DUMP_STATES only the columns of a fixed,
    seeded sample of DUMP_STATES state indices (increasing) are written: 2 x 7 x 2^18 doubles = 29 MB for the FR3 step."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    for name, x in arrays.items():
        if x.shape[1] > DUMP_STATES:
            idx = np.sort(np.random.default_rng(DUMP_SEED).choice(x.shape[1], DUMP_STATES, replace=False))
            x = x.index_select(1, torch.from_numpy(idx).to(x.device))
        np.save(os.path.join(out_dir, name + ".npy"), x.cpu().numpy())


def run_ours(args, rank, local_rank, world):
    import torch
    import torch.distributed as dist
    import rigidbody_rs_b200 as rb
    from rigidbody_rs_b200.shard import max_over_ranks, shard_bounds, sum_over_ranks

    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    mb = rb.Multibody.from_urdf(os.path.join(ROOT, "assets", "fr3.urdf"), device=local_rank)
    n, B = mb.n, args.states
    lim = mb.limits()
    first = rank * B                                   # each rank samples its own slice of the global index space
    q = torch.empty((n, B), dtype=torch.float64, device=dev)
    dq, ddq, tau_in = torch.empty_like(q), torch.empty_like(q), torch.empty_like(q)
    tau, qdd = torch.empty_like(q), torch.empty_like(q)
    mb.fill(q, SEED_RNEA, 0, lim["lower"], lim["upper"], first)
    mb.fill(dq, SEED_RNEA, 1, -lim["velocity"], lim["velocity"], first)
    mb.fill(ddq, SEED_RNEA, 2, -10.0, 10.0, first)
    mb.fill(tau_in, SEED_FD, 3, -lim["effort"], lim["effort"], first)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        """max-over-ranks device time per call of fn (CUDA events on the launching stream, barrier on both sides)."""
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        return max_over_ranks(e0.elapsed_time(e1) / steps, dev)

    # ------------------------------------------------------------------ headline: RNEA launch + FD launch, K steps
    for _ in range(args.warmup):
        mb.rnea(q, dq, ddq, out=tau)
        mb.forward_dynamics(q, dq, tau_in, out=qdd)
    K = args.steps
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(K)]
    sampler = ClockSampler(local_rank); sampler.start()
    barrier()
    launches0 = mb.launch_count
    t_start = torch.cuda.Event(enable_timing=True); t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    for k in range(K):
        ev[k][0].record()
        mb.rnea(q, dq, ddq, out=tau)
        ev[k][1].record()
        mb.forward_dynamics(q, dq, tau_in, out=qdd)
        ev[k][2].record()
    t_end.record()
    barrier()
    clocks = sampler.stop()
    launches = mb.launch_count - launches0
    mb.sync()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, {"tau": tau, "qdd": qdd})
    total_ms = t_start.elapsed_time(t_end)
    # FP64 roofline denominator: DFMA probe on the same GPU in the same run, run for about as long as the timed
    # region (a burst of a few ms keeps 1965 MHz; seconds of FP64 work pull ~1 kW and settle near 1.7 GHz under
    # sw_power_cap), so burst numbers are divided by a burst peak and sustained numbers by a sustained peak
    probe_ms = int(min(2000.0, max(10.0, total_ms)))
    fp64_peak = mb.fp64_peak_tflops(probe_ms)
    peak_note = f"DFMA probe (multibody_gpu_measure_fp64_peak) on this GPU in this run, {probe_ms} ms; nominal 148 x 64 x 2 x 1.965 GHz = 37.2"
    ms_step = max_over_ranks(total_ms / K, dev)
    ms_rnea = max_over_ranks(sum(e[0].elapsed_time(e[1]) for e in ev) / K, dev)
    ms_fd = max_over_ranks(sum(e[1].elapsed_time(e[2]) for e in ev) / K, dev)
    units = sum_over_ranks(2.0 * B, dev)               # evaluations all ranks processed per step
    value = units / (ms_step * 1e-3)
    hbm_peak, hbm_src = measured_peaks()
    fr3 = mb.kernel_variant == "fr3-specialised"

    def roof(kernel, alg_flops, ms):
        pr = profiled(kernel)
        full = B == STATES_PER_GPU and pr is not None
        instr, src, fl = FP64_INSTR[kernel], "static SASS count minus the out-of-range sin/cos fallback (tools/sass_count.sh)", None
        if full and "fp64_thread_instr" in pr:
            instr, src, fl = pr["fp64_thread_instr"] / B, "ncu sm__inst_executed_pipe_fp64.sum x 32 / states (" + pr["source"] + ")", pr["fp64_thread_flops"] / B
        return fp64_roofline(kernel, ms, float(B), instr if fr3 else float("nan"), fl, alg_flops, BYTES_PER_EVAL, fp64_peak, peak_note,
                             hbm_peak, hbm_src, pr["bytes"] if full else None, pr["source"] if full else None, src)

    # ------------------------------------------------------------------ configs.fused_rnea_fd: one pass, both results
    both = torch.empty((2 * n, B), dtype=torch.float64, device=dev)
    ms_fused = timed(lambda: mb.rnea_fd(q, dq, ddq, tau_in, out=both), K, args.warmup)
    fused_ok = bool(torch.equal(both[n:, :65536], qdd[:, :65536])) and \
        float(((both[:n, :65536] - tau[:, :65536]).abs().amax(0) / tau[:, :65536].abs().amax(0).clamp_min(1.0)).max()) < 1e-12
    pr = profiled("rb_rnea_fd_kernel")
    fused_instr = pr["fp64_thread_instr"] / STATES_PER_GPU if pr and "fp64_thread_instr" in pr else 1348.0 - 126.0
    cfg_fused = {"value": units / (ms_fused * 1e-3), "unit": UNIT, "ms_per_step": ms_fused, "scaling": "weak",
                 "step": "1 rb_rnea_fd_kernel launch: tau = rnea(q, dq, ddq) AND qdd = fd(q, dq, tau_in) of the same 2^24 states "
                         "(shared sin/cos, bias recursion and mass matrix; tau = bias + H ddq)",
                 "matches_separate_kernels": fused_ok,
                 "roofline": fp64_roofline("rb_rnea_fd_kernel", ms_fused, float(B), fused_instr, pr.get("fp64_thread_flops", 0) / STATES_PER_GPU if pr else None,
                                           RNEA_FLOPS + FD_FLOPS, 336.0, fp64_peak, peak_note, hbm_peak, hbm_src,
                                           pr["bytes"] if pr and B == STATES_PER_GPU else None, pr["source"] if pr else None)}
    del both

    # ------------------------------------------------------------------ end to end through the C ABI with HOST buffers
    Be = args.e2e_states
    hq, hdq, hddq, htau_in = (rb.host_empty((n, Be)) for _ in range(4))
    htau, hqdd = rb.host_empty((n, Be)), rb.host_empty((n, Be))
    for h, d in ((hq, q), (hdq, dq), (hddq, ddq), (htau_in, tau_in)):
        h[...] = d[:, :Be].cpu().numpy()
    e2e_steps = max(1, min(K, args.e2e_steps))
    mb.rnea(hq, hdq, hddq, out=htau); mb.forward_dynamics(hq, hdq, htau_in, out=hqdd)      # warm-up (allocates staging)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        mb.rnea(hq, hdq, hddq, out=htau)
        mb.forward_dynamics(hq, hdq, htau_in, out=hqdd)
    torch.cuda.synchronize()
    sep_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / e2e_steps, dev)
    # the same step through the one-call entry point (multibody_rnea_fd_batch): q and dq cross PCIe once instead of
    # twice (4 input arrays instead of 6) and the fused kernel serves every chunk -- the bus is what bounds this number
    hout = rb.host_empty((2 * n, Be))
    mb.rnea_fd(hq, hdq, hddq, htau_in, out=hout)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        mb.rnea_fd(hq, hdq, hddq, htau_in, out=hout)
    torch.cuda.synchronize()
    e2e_ms = max_over_ranks((time.perf_counter() - t0) * 1e3 / e2e_steps, dev)
    e2e_units = sum_over_ranks(2.0 * Be, dev)
    up_b, down_b = 4 * n * Be * 8, 2 * n * Be * 8
    # the host results equal the device-resident ones: qdd bit for bit, tau to rounding (fused kernel)
    same = bool(np.array_equal(htau[:, :4096], tau[:, :4096].cpu().numpy())) and bool(np.array_equal(hout[n:], hqdd)) \
        and float(np.abs(hout[:n] - htau).max() / max(1.0, np.abs(htau).max())) < 1e-12
    # the ceiling: the same bytes, both directions at once, pinned memory, no kernel -- every rank at the same time.
    # Buffers are allocated and warmed BEFORE the barrier: pinning 4 GB takes about a second and the ranks' allocations
    # serialise in the kernel, so a probe that allocates inside its timed call (multibody_gpu_measure_copy_peak, round 2's
    # first version) let the ranks' passes drift apart until nobody competed with anybody -- 215 GB/s "ceilings" for 8
    # processes on a host whose DRAM serves about 100 GB/s of H2D next to 50 GB/s of D2H.
    ceil_ms = max_over_ranks(bare_copy_ms(up_b, down_b, 3, dev, barrier), dev)
    e2e = {"value": e2e_units / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": up_b, "d2h_bytes_per_step": down_b,
           "states_per_gpu": Be, "steps": e2e_steps, "ms_per_step": e2e_ms,
           "h2d_GBs": world * up_b / e2e_ms / 1e6, "d2h_GBs": world * down_b / e2e_ms / 1e6,
           "copy_ceiling": {"h2d_GBs": world * up_b / ceil_ms / 1e6, "d2h_GBs": world * down_b / ceil_ms / 1e6, "ms_per_step": ceil_ms,
                            "evals_per_s": e2e_units / (ceil_ms * 1e-3),
                            "how": "the same bytes per direction from / to pinned host memory (buffers of up to 2 GiB walked front to back, "
                                   "64 MiB copies, two streams: both directions at once), no kernel; buffers pinned before a barrier, then all "
                                   "ranks copy at the same time; max over ranks of the mean pass"},
           "frac_of_copy_ceiling": ceil_ms / e2e_ms,
           "api": "Multibody.rnea_fd on pinned numpy arrays -> multibody_rnea_fd_batch(RB_MEM_HOST), one process per GPU: q, dq, ddq, tau_in up, tau and qdd down",
           "matches_device_path": same,
           "separate_calls": {"value": e2e_units / (sep_ms * 1e-3), "ms_per_step": sep_ms, "h2d_bytes_per_step": 6 * n * Be * 8,
                              "api": "Multibody.rnea + Multibody.forward_dynamics -> multibody_{rnea,forward_dynamics}_batch(RB_MEM_HOST)"}}
    for h in (hq, hdq, hddq, htau_in, htau, hqdd, hout):
        rb.host_free(h)
    del hq, hdq, hddq, htau_in, htau, hqdd, hout

    # one process, one handle, all N GPUs: multibody_gpu_new_multi cuts ONE host batch into N contiguous slices (rank 0
    # drives it while the other ranks wait at the barrier); its own bare-copy ceiling beside it
    if world > 1:
        barrier()
        if rank == 0:
            Bm = (1 << 22) * world
            mm = rb.Multibody.from_urdf(os.path.join(ROOT, "assets", "fr3.urdf"), devices=list(range(world)))
            mq, mdq, mddq, mtin = (rb.host_empty((n, Bm)) for _ in range(4))
            mout = rb.host_empty((2 * n, Bm))
            rng = np.random.default_rng(0)
            for h, (lo_, hi_) in zip((mq, mdq, mddq, mtin), ((lim["lower"], lim["upper"]), (-lim["velocity"], lim["velocity"]), (-10.0, 10.0), (-lim["effort"], lim["effort"]))):
                h[...] = (np.broadcast_to(lo_, (n,))[:, None] + (np.broadcast_to(hi_, (n,)) - np.broadcast_to(lo_, (n,)))[:, None] * rng.random((1, Bm)))
            mm.rnea_fd(mq, mdq, mddq, mtin, out=mout)
            ts = []
            for _ in range(e2e_steps):
                t0 = time.perf_counter(); mm.rnea_fd(mq, mdq, mddq, mtin, out=mout); ts.append(time.perf_counter() - t0)
            msec = sum(ts) / len(ts)
            mu, md = mm.copy_peak(4 * n * Bm * 8, 2 * n * Bm * 8, 2)
            e2e["single_process_multi_device"] = {
                "value": 2.0 * Bm / msec, "unit": UNIT, "ms_per_step": msec * 1e3, "states": Bm, "devices": world,
                "h2d_GBs": 4 * n * Bm * 8 / msec / 1e9, "d2h_GBs": 2 * n * Bm * 8 / msec / 1e9,
                "copy_ceiling": {"h2d_GBs": mu, "d2h_GBs": md, "evals_per_s": 2.0 * Bm / (4 * n * Bm * 8 / mu / 1e9)},
                "frac_of_copy_ceiling": (4 * n * Bm * 8 / mu / 1e9) / msec,
                "api": "multibody_gpu_new_multi over all GPUs, ONE multibody_rnea_fd_batch(RB_MEM_HOST) call on one pinned host batch; "
                       "the other ranks idle"}
            for h in (mq, mdq, mddq, mtin, mout):
                rb.host_free(h)
            mm.close()
        barrier()

    # optional assembly of the sharded result on every rank: ONE NCCL all-gather of tau (SURVEY 8e), outside the timed
    # region and reported separately -- the compute path itself exchanges nothing
    gather = None
    if world > 1:
        Bg = min(B, 1 << 22)                              # 235 MB per rank: enough to see the NVLink rate
        part = tau[:, :Bg].contiguous()
        full = torch.empty((world, n, Bg), dtype=torch.float64, device=dev)
        dist.all_gather_into_tensor(full, part)           # warm-up (communicator set-up)
        torch.cuda.synchronize()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        barrier()
        g0.record()
        dist.all_gather_into_tensor(full, part)
        g1.record()
        torch.cuda.synchronize()
        gms = max_over_ranks(g0.elapsed_time(g1), dev)
        ok_g = bool(torch.equal(full[rank], part))
        gather = {"collective": "ncclAllGather(tau)", "ms": gms, "bytes_per_rank": int(part.numel() * 8),
                  "recv_GB_per_s_per_rank": (world - 1) * part.numel() * 8 / (gms * 1e-3) / 1e9, "own_slice_intact": ok_g}
        del full, part

    # ------------------------------------------------------------------ configs.rollout: BASELINE configs[3], strong scaling
    Ht, dt = 64, 1e-3
    lo, hi = shard_bounds(65536, world, rank)
    Bt = hi - lo
    q0, dq0 = torch.empty((n, Bt), dtype=torch.float64, device=dev), torch.empty((n, Bt), dtype=torch.float64, device=dev)
    mb.fill(q0, 0x5EED0003, 0, lim["lower"], lim["upper"], lo)
    mb.fill(dq0, 0x5EED0003, 1, -lim["velocity"], lim["velocity"], lo)
    taus = torch.empty((Ht, n, Bt), dtype=torch.float64, device=dev)
    for t in range(Ht):
        mb.fill(taus[t], 0x5EED0003, 4 + t % 32, -lim["effort"], lim["effort"], t * 65536 + lo)
    l0 = mb.launch_count
    ms_ro = timed(lambda: mb.rollout(q0, dq0, taus, dt), max(3, min(K, 10)), 3)
    ro_launches = mb.launch_count - l0
    ro_units = sum_over_ranks(float(Bt * Ht), dev)
    pr = profiled("rb_rollout_kernel")
    ro_instr = pr["fp64_thread_instr"] / (65536 * Ht) if pr and "fp64_thread_instr" in pr else FP64_INSTR["rb_fd_kernel"] + 14.0
    cfg_rollout = {"metric": "FR3 MPC rollout FD steps/sec (fp64)", "value": ro_units / (ms_ro * 1e-3), "unit": "steps/s", "ms_per_step": ms_ro,
                   "scaling": "strong", "trajectories": 65536, "trajectories_per_gpu": Bt, "horizon": Ht, "dt": dt,
                   "step": "1 rb_rollout_kernel launch: semi-implicit Euler through forward dynamics, (q, dq) written after every step",
                   "roofline": fp64_roofline("rb_rollout_kernel", ms_ro, float(Bt * Ht), ro_instr, pr.get("fp64_thread_flops", 0) / (65536 * Ht) if pr else None,
                                             FD_FLOPS + 28.0, 168.0, fp64_peak, peak_note, hbm_peak, hbm_src,
                                             pr["bytes"] if pr and world == 1 else None, pr["source"] if pr else None,
                                             "ncu op counters" if pr and "fp64_thread_instr" in pr else "FD kernel count + 14 (Euler update)")}
    del q0, dq0, taus

    # ------------------------------------------------------------------ configs.chain32: BASELINE configs[4], strong scaling
    cfg_chain32 = None
    if not args.no_chain32:
        del q, dq, ddq, tau_in, tau, qdd
        torch.cuda.empty_cache()
        mc = rb.Multibody.from_urdf(os.path.join(ROOT, "assets", "chain32.urdf"), device=local_rank)
        lo, hi = shard_bounds(args.chain32_states, world, rank)
        Bc, nc = hi - lo, mc.n
        pi = np.full(nc, np.pi)
        cq = torch.empty((nc, Bc), dtype=torch.float64, device=dev)
        cdq, cx, cin, co1, co2 = (torch.empty_like(cq) for _ in range(5))
        mc.fill(cq, 0x5EED0005, 0, -pi, pi, lo)
        mc.fill(cdq, 0x5EED0005, 1, -2.0, 2.0, lo)
        mc.fill(cx, 0x5EED0005, 2, -10.0, 10.0, lo)
        mc.fill(cin, 0x5EED0005, 3, -50.0, 50.0, lo)
        e = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        mc.rnea(cq, cdq, cx, out=co1); mc.forward_dynamics(cq, cdq, cin, out=co2)
        barrier()
        ksteps = 2
        tr = tf = 0.0
        for _ in range(ksteps):
            e[0].record(); mc.rnea(cq, cdq, cx, out=co1); e[1].record(); mc.forward_dynamics(cq, cdq, cin, out=co2); e[2].record()
            torch.cuda.synchronize()
            tr += e[0].elapsed_time(e[1]); tf += e[1].elapsed_time(e[2])
        barrier()
        ms_cr, ms_cf = max_over_ranks(tr / ksteps, dev), max_over_ranks(tf / ksteps, dev)
        c_units = sum_over_ranks(2.0 * Bc, dev)
        prf, prr = profiled("rbq_fd_kernel"), profiled("rb_long_rnea_kernel")

        def scaled(pr_):      # DRAM bytes of this launch, scaled per state from the committed 2^20-state capture
            return (pr_["bytes"] / (1 << 20) * Bc, pr_["source"] + f" (per state, x {Bc} states)") if pr_ else (None, None)
        cfg_chain32 = {"metric": "chain32 RNEA+FD evals/sec (fp64)", "value": c_units / ((ms_cr + ms_cf) * 1e-3), "unit": UNIT,
                       "ms_per_step": ms_cr + ms_cf, "scaling": "strong", "states": args.chain32_states, "states_per_gpu": Bc, "n_joints": nc,
                       "kernel_variant": mc.kernel_variant, "step": "1 rb_long_rnea_kernel launch + 1 rbq_fd_kernel launch over all states",
                       "roofline": fp64_roofline("rbq_fd_kernel", ms_cf, float(Bc), prf["fp64_thread_instr"] / (1 << 20) if prf and "fp64_thread_instr" in prf else 908.0 * 32,
                                                 prf["fp64_thread_flops"] / (1 << 20) if prf and "fp64_thread_flops" in prf else None,
                                                 53800.0, 1024.0, fp64_peak, peak_note, hbm_peak, hbm_src, *scaled(prf),
                                                 "FP64-pipe instruction slots per state: warp instructions x 32 lanes / states of the capture (8 lanes own a state in "
                                                 "the matrix phase, 16 in the chain phase; idle triangle lanes count as used slots)"),
                       "roofline_rnea": fp64_roofline("rb_long_rnea_kernel", ms_cr, float(Bc), prr["fp64_thread_instr"] / (1 << 20) if prr and "fp64_thread_instr" in prr else 3626.0,
                                                      prr["fp64_thread_flops"] / (1 << 20) if prr and "fp64_thread_flops" in prr else None,
                                                      9476.0, 1024.0, fp64_peak, peak_note, hbm_peak, hbm_src, *scaled(prr))}
        del cq, cdq, cx, cin, co1, co2

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": args.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f64", "data": "synthetic",
        "config": {"workload": "fr3_rnea+fd_16M", "states_per_gpu": B, "n_joints": n, "layout": "soa",
                   "kernel_variant": mb.kernel_variant, "cache": "inputs larger than L2 (2.8 GB read per kernel)",
                   "step": "1 RNEA launch + 1 forward-dynamics launch over all states", "parallelism": f"dp{world}"},
        "roofline": roof("rb_fd_kernel", FD_FLOPS, ms_fd),
        "roofline_rnea": roof("rb_rnea_kernel", RNEA_FLOPS, ms_rnea),
        "configs": {"fused_rnea_fd": cfg_fused, "rollout": cfg_rollout, "chain32": cfg_chain32},
        "e2e": e2e,
        "gpu_launches": int(launches), "clocks": clocks,
    }
    line["configs"]["rollout"]["gpu_launches"] = int(ro_launches)
    if gather is not None:
        line["gather"] = gather
    if rank == 0 and world == 1 and not args.no_cpu:
        cb, _, _ = cpu_arm(None, 2, 1)
        line["cpu_baseline"] = cb
    elif rank == 0:
        line["cpu_baseline"] = None
    if rank == 0:
        print(json.dumps(line), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--states", type=int, default=STATES_PER_GPU, help="states per GPU per step")
    ap.add_argument("--e2e-states", type=int, default=STATES_PER_GPU, help="states per GPU per end-to-end step")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-chain32", action="store_true", help="skip the configs.chain32 leg")
    ap.add_argument("--chain32-states", type=int, default=1 << 26, help="states of the chain32 leg, split over the GPUs (BASELINE configs[4]: 64M)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write DIR/tau.npy and DIR/qdd.npy: the last step's RNEA and forward-dynamics "
                         "results, float64 [n, S], S = a fixed seeded sample of 2^18 states (all if fewer); rank 0's states")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank)
        return
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the engine has no CPU fallback (use --impl reference for the CPU arm)")
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, local_rank, world)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
