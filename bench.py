#!/usr/bin/env python
"""bench.py -- cell-layer updates/s of the msqg timestep (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one full predictor-corrector timestep (2 x (PV inversion + RHS +
stage update)) of the 4096^2 x nl=4 synthetic double-gyre workload of
SURVEY.md 8(d).  `value` is measured with the state resident in HBM; `e2e` is
the same step driven through the C ABI with HOST buffers (q uploaded from and
downloaded to pinned host memory every step).  `--impl reference` times the
CPU oracle (the reference itself cannot be built here: Basilisk/qcc absent) on
all host cores on the same workload.

`--dump-outputs DIR` writes, after the K timed steps, what the timed path returned
in its last step as DIR/<name>.npy (float64): `dt` and `t` (the last time step and
the model time after it) and `psi` and `q` (the stream function and potential
vorticity, flattened [layer][y][x]; fields of more than DUMP_SAMPLE values are cut
to a fixed seeded sample, see dump_indices).  Inputs are synthetic and seeded, so
two builds run with the same arguments can be compared file for file.  (The
`--impl reference` sweep is an OpenMP loop whose result depends on thread timing;
its outputs repeat from run to run with OMP_NUM_THREADS=1 only.)
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True  # the benchmark leaves the tree it runs from as it found it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

METRIC = "cell-layer updates/s"
UNIT = "cell-layer updates/s"
N_DEFAULT, NL_DEFAULT = 4096, 4


MODAL = False  # --modal: MODE_PV_INVERT 1 (BASELINE config 3), set by main()


PERIODIC = False  # --periodic: sbc = -1 (doubly periodic domain, datapoint only)
VARRO = False  # --varRo: Ro(y) (horizontally varying stretching / vertical modes, datapoint only)


def workload_kw(N, nl):
    from common import base_kw
    over = {}
    if MODAL:
        over["mode_pv_invert"] = 1
    if PERIODIC:
        over["sbc"] = -1.
    if VARRO:
        over["varRo"] = 1
    return base_kw(N, nl, **over)


def workload_psi(N, nl):
    from common import synth_psi, periodic_psi
    return periodic_psi(N, nl) if PERIODIC else synth_psi(N, nl)


def workload_name(N, nl):
    return "msqg double-gyre %d^2 x nl=%d, %s, tolerance 1e-3%s%s" % (
        N, nl, "vertical-mode inversion (MODE_PV_INVERT 1)" if MODAL else "layer-coupled multigrid inversion (MODE_PV_INVERT 0)",
        ", doubly periodic (sbc = -1)" if PERIODIC else "", ", Ro(y) (varRo = 1)" if VARRO else "")


DUMP_SAMPLE = 1 << 21  # values kept per field by --dump-outputs (16 MB in float64; psi + q stay well under 64 MB)


def dump_indices(n):
    """Flat indices of a field of n values that --dump-outputs keeps: all of them up to DUMP_SAMPLE, else a sorted
    sample drawn without replacement from a fixed seed, so runs with the same arguments keep the same cells."""
    if n <= DUMP_SAMPLE:
        return np.arange(n)
    return np.sort(np.random.default_rng(0).choice(n, DUMP_SAMPLE, replace=False))


def dump_outputs(d, dt, t, psi, q):
    """--dump-outputs: the last timed step's dt and model time t, and psi and q (sampled by dump_indices)"""
    os.makedirs(d, exist_ok=True)
    psi, q = np.ravel(psi), np.ravel(q)
    idx = dump_indices(psi.size)
    for name, a in (("dt", np.ravel(dt)), ("t", np.ravel(t)), ("psi", psi[idx]), ("q", q[idx])):
        np.save(os.path.join(d, name + ".npy"), np.asarray(a, dtype=np.float64))


def algorithmic_bytes(nl):
    """SURVEY.md 8(d): bytes per cell-layer of each piece (F = 8 B, sigma = (nl-1)/nl)."""
    sig = (nl - 1.0) / nl
    return dict(relax_sweep=(3 + sig) * 8, residual=(3 + sig) * 8, restrict=5.0 / 3 * 8, prolong=5.0 / 3 * 8,
                correct=3 * 8.0, rhs=(5 + sig) * 8)


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML in a thread (every 5 ms; a step is ~10-20 ms),
    nvidia-smi as a fallback."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.nv = index, [], None, None
        self.sm, self.reasons, self.mx, self.stop_flag = [], set(), None, False
        try:
            import pynvml
            pynvml.nvmlInit()
            idx = index
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            if vis:
                try:
                    idx = int(vis.split(",")[index])
                except Exception:
                    idx = index
            self.h = pynvml.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
            self.nv = pynvml
        except Exception:
            self.nv = None

    def _nvml_loop(self):
        nv = self.nv
        bits = {"hw_slowdown": getattr(nv, "nvmlClocksEventReasonHwSlowdown", 0x8),
                "hw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                "sw_thermal_slowdown": getattr(nv, "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                "sw_power_cap": getattr(nv, "nvmlClocksEventReasonSwPowerCap", 0x4)}
        get_reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or getattr(nv, "nvmlDeviceGetCurrentClocksThrottleReasons")
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
                r = int(get_reasons(self.h))
                for name, bit in bits.items():
                    if r & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.005)

    def start(self):
        if self.nv is not None:
            self.th = threading.Thread(target=self._nvml_loop, daemon=True)
            self.th.start()
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.nv is not None:
            self.stop_flag = True
            self.th.join(timeout=1)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx,
                    "reasons": sorted(self.reasons), "samples": len(self.sm), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace(".", "").isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 9:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm), "source": "nvidia-smi"}


def cpu_oracle_run(N, nl, steps, warmup, smoother="lex", dump=None):
    """The CPU oracle built with OpenMP (same algorithm and loop order as the reference,
    foreach() as an omp-for like `qcc -fopenmp`), on all host cores.  dump: --dump-outputs directory or None."""
    from oracle import oracle as O
    cores = os.cpu_count() or 1
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    m = O.Model(O.make_params(omp=True, **workload_kw(N, nl)), omp=True)
    m.set_smoother(smoother)
    m.set(O.PSI, workload_psi(N, nl))
    m.set_const()
    for _ in range(warmup):
        m.step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step_dt = m.step()
    dt = time.perf_counter() - t0
    cyc = m.L.orc_total_cycles(m.h)
    if dump:
        dump_outputs(dump, step_dt, m.t, m.get(O.PSI), m.get(O.Q))
    m.close()
    return N * N * nl * steps / dt, dt / steps * 1e3, int(os.environ["OMP_NUM_THREADS"]), cyc


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    # torchrun pins OMP_NUM_THREADS=1 for its workers when the variable is unset; the reference arm runs on rank 0 alone
    # and is meant to use every host core, so that default is undone here (an explicit user setting > 1 is kept)
    if os.environ.get("OMP_NUM_THREADS", "1") == "1" and "TORCHELASTIC_RUN_ID" in os.environ:
        os.environ["OMP_NUM_THREADS"] = str(cores)
    # the SAME configuration as our arm: the full args.N^2 x nl grid (4096^2 x 4: a few seconds per step on 16+ cores),
    # the reference's own sweep (lexicographic, foreach() as an omp-for), --steps timed steps after at most one warm-up
    # step (the CPU takes seconds per step).
    rsteps, rwarm = args.steps, max(0, min(args.warmup, 1))
    val, ms, threads, _ = cpu_oracle_run(args.N, args.nl, rsteps, rwarm, "lex", dump=args.dump_outputs)
    sample = ("the full %d^2 x nl=%d workload, %d timed steps after %d warm-up (warm-up bounded: the CPU takes seconds per step)"
              % (args.N, args.nl, rsteps, rwarm))
    line = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": workload_name(args.N, args.nl), "N": args.N, "nl": args.nl,
                       "timed_steps": rsteps,
                       "reference": "CPU oracle (C restatement of msqg with the reference's lexicographic sweep, OpenMP; "
                                    "the Basilisk build itself needs qcc, absent here)"},
            "cpu_baseline": {"value": val, "unit": UNIT, "cores": threads, "kind": "port", "sample": sample},
            "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def run_ensemble(args):
    """BASELINE config 5: stochastic ensemble, `--members` members per GPU of 512^2 x nl=3 (32 members on 8 GPUs), replicas
    only: no communication between members.  Aggregate cell-layer updates/s over all members and GPUs."""
    import torch
    import torch.distributed as dist
    from msom_b200 import capi as G
    from msom_b200.ensemble import Ensemble
    from common import base_kw, synth_psi
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    N, nl, M = args.ens_N, 3, args.members
    kw = base_kw(N, nl, stochastic=1, tr_stoch=10., amp_stoch=1.)
    ens = Ensemble(G.make_params(**kw), M, local, seeds=[1000 + rank * M + i for i in range(M)], noise=args.noise, smoother=args.smoother)
    ens.set(G.PSI, synth_psi(N, nl)); ens.set(G.SSTOCH, np.full((nl, N, N), 1e-3)); ens.set_const()
    ens.step(max(args.warmup, 3))
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    step_dts = ens.step(args.steps)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([dt], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
    if args.dump_outputs:   # one value of dt and t per member, psi and q stacked [member][layer][y][x]
        dump_outputs(args.dump_outputs, [d[-1] for d in step_dts],
                     [ens.L.msqg_ensemble_time(ens.h, k) for k in range(len(ens))], ens.get(G.PSI), ens.get(G.Q))
    cycles = sum(m.total_cycles for m in ens.members)
    launches = sum(m.launches for m in ens.members)
    ens.close()
    if rank == 0:
        val = float(N) * N * nl * M * world * args.steps / dt
        line = {"metric": METRIC, "value": val, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
                "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "f64", "data": "synthetic",
                "config": {"workload": "msqg qg_stochastic ensemble, %d members x %d^2 x nl=%d per GPU (BASELINE config 5), noise=%s, smoother=%s"
                                       % (M, N, nl, args.noise, args.smoother),
                           "members_total": M * world, "parallelism": "replicas: %d member(s) per GPU on own streams, no communication" % M,
                           "timing": "wall clock around the concurrent member steps (device-synchronised on both sides), max over ranks"},
                "gpu_launches": int(launches)}
        os.write(real_stdout, (json.dumps(line) + "\n").encode())
    if world > 1:
        dist.destroy_process_group()


def run_ours(args):
    import torch
    import torch.distributed as dist
    from msom_b200 import capi as G
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the msqg timestep has no CPU path")
    torch.cuda.set_device(local)
    # rank 0 prints ONE JSON line: anything a library writes to fd 1 meanwhile (NCCL's version banner ...) goes to stderr
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        os.write(real_stdout, (json.dumps(obj) + "\n").encode())

    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    N, nl = args.N, args.nl
    cells = float(N) * N * nl

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    def allmax(x):
        if world == 1:
            return x
        t = torch.tensor([x], device="cuda", dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    sm = args.smoother
    if world == 1:
        m = G.Model(G.make_params(**workload_kw(N, nl)), local)
        m.set_smoother(sm)
        stream = torch.cuda.Stream(device=local)
        m.set_stream(stream.cuda_stream)
        m.set(G.PSI, workload_psi(N, nl))
        m.set_const()
        step = m.step
        parallelism = "1 GPU"
    else:
        # strong scaling: the SAME N^2 x nl grid cut into px x py tiles, one per GPU.  rb: deep-halo exchange once per
        # level and cycle (grouped ncclSend/ncclRecv to the 8 neighbours), levels below agg_n replicated on every GPU
        # (ncclAllGather of the restricted residual); results identical to the 1-GPU run bit for bit.
        from msom_b200.dist import nccl_group
        m = nccl_group(G.make_params(**workload_kw(N, nl)), args.agg_n, local, smoother=sm)
        m.set_global(G.PSI, workload_psi(N, nl))
        m.set_const()
        step = m.step
        if sm == "rb":
            parallelism = ("%dx%d tiles, one deep-halo exchange per level and cycle (%s), levels < %d replicated on every GPU "
                           "(ncclAllGather), residual norm by ncclAllReduce" % (m.px, m.py, m.transport, args.agg_n))
        else:
            parallelism = "%dx%d tiles, NCCL halo exchange per sweep, levels < %d agglomerated on rank 0" % (m.px, m.py, args.agg_n)

    for _ in range(args.warmup):
        step()
    # ---- timed region: K steps, state resident in HBM (CUDA events on the stream the kernels are launched on)
    barrier()
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    c0, l0 = m.total_cycles, m.launches
    if world == 1:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            for _ in range(args.steps):
                step_dt = step()
            e1.record(stream)
        e1.synchronize()
        ms_total = e0.elapsed_time(e1)
    else:
        m.timer_start()
        for _ in range(args.steps):
            step()
        ms_total = m.timer_stop()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    cycles, launches = m.total_cycles - c0, m.launches - l0
    if args.dump_outputs:   # before the untimed passes below advance the state further
        dump_outputs(args.dump_outputs, step_dt, m.t, m.get(G.PSI), m.get(G.Q))
    ms_total = allmax(ms_total)
    ms_step = ms_total / args.steps
    value = N * N * nl * args.steps / (ms_total * 1e-3)
    # ---- per-kernel device times: a second, untimed pass of the same steps with per-launch events on the same stream
    # (the library replays recorded CUDA graphs in the timed region; with events between the launches it issues them
    # one by one, so this pass is slightly slower than the timed one and is used for shares and per-launch times only)
    psteps = max(1, min(args.steps, 5))
    m.profile(True)
    pc0 = m.total_cycles
    for _ in range(psteps):
        step()
    prof = m.profile_read()
    m.profile(False)
    pcycles = m.total_cycles - pc0
    prof_ms_total = sum(v["ms"] for v in prof.values())
    barrier()

    # ---- end to end through the C ABI with host buffers: every step takes its q from pinned host memory and returns
    # its q to pinned host memory.
    #   serial:    msqg_set_field; step; msqg_get_field (the transfers and the step follow each other)
    #   pipelined: msqg_set_field_async / _commit / msqg_get_field_async (include/msqg.h): the upload of the next state
    #              and the download of the previous result run on their own streams while a state is stepped -- the
    #              loop of a caller that advances a stream of independent states (ensemble members, BFN sweeps).
    #              Same bytes per step; the headline `e2e` is this loop, `e2e.serial` keeps the other one.
    esteps = max(1, min(args.steps, 5))
    if world == 1:
        tile_shape, getq, setq = (nl, N, N), (lambda a: G.check(m.L.msqg_get_field(m.h, G.Q, a))), \
            (lambda a: G.check(m.L.msqg_set_field(m.h, G.Q, a)))
        tile_h = m.h
    else:
        _, _, _, _, tnx, tny = m.boxes[0]
        tile_shape = (nl, tny, tnx)
        getq = lambda a: G.check(m.L.msqg_group_get_field(m.h, 0, G.Q, a))
        setq = lambda a: G.check(m.L.msqg_group_set_field(m.h, 0, G.Q, a))
        tile_h = m.L.msqg_group_tile(m.h, 0)
        G.lib()  # binds the argtypes of the single-model entry points used on the tile handle below
    hq = torch.empty(tile_shape, dtype=torch.float64).pin_memory()
    hq_np = hq.numpy()
    getq(hq_np)
    barrier()
    t0 = time.perf_counter()
    for _ in range(esteps):
        setq(hq_np)
        step()
        getq(hq_np)
    torch.cuda.synchronize()
    e2e_serial_s = allmax(time.perf_counter() - t0)
    e2e_serial_val = N * N * nl * esteps / e2e_serial_s
    psteps_io = max(esteps, args.steps)
    LG = G.lib()
    hin = [torch.empty(tile_shape, dtype=torch.float64).pin_memory() for _ in range(2)]
    hout = [torch.empty(tile_shape, dtype=torch.float64).pin_memory() for _ in range(2)]
    for h in hin:
        h.copy_(hq)
    hin_np, hout_np = [h.numpy() for h in hin], [h.numpy() for h in hout]
    # one untimed pass of the loop body: the first transfer allocates the staging buffers, streams and events
    G.check(LG.msqg_set_field_async(tile_h, G.Q, hin_np[0]))
    G.check(LG.msqg_set_field_commit(tile_h))
    step()
    G.check(LG.msqg_get_field_async(tile_h, G.Q, hout_np[0]))
    G.check(LG.msqg_io_wait(tile_h))
    torch.cuda.synchronize()
    barrier()
    t0 = time.perf_counter()
    G.check(LG.msqg_set_field_async(tile_h, G.Q, hin_np[0]))
    for k in range(psteps_io):
        G.check(LG.msqg_set_field_commit(tile_h))
        if k + 1 < psteps_io:
            G.check(LG.msqg_set_field_async(tile_h, G.Q, hin_np[(k + 1) & 1]))
        step()
        G.check(LG.msqg_get_field_async(tile_h, G.Q, hout_np[k & 1]))
    G.check(LG.msqg_io_wait(tile_h))
    torch.cuda.synchronize()
    e2e_s = allmax(time.perf_counter() - t0)
    e2e_val = N * N * nl * psteps_io / e2e_s
    if not np.isfinite(hout_np[(psteps_io - 1) & 1]).all():
        raise RuntimeError("pipelined e2e loop returned a non-finite field")
    tile_cells = float(np.prod(tile_shape))
    if rank != 0:
        if world > 1:
            m.close()
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel: finest-level relax launches
    ab = algorithmic_bytes(nl)
    peak, peak_src = peaks()
    rf = prof["relax_fine"]
    roof = None
    if rf["count"] > 0 and rf["ms"] > 0:
        alg_bytes_per_launch = ab["relax_sweep"] * tile_cells * (rf["aux"] / rf["count"])
        if MODAL:  # one launch relaxes ONE vertical mode: scalar Helmholtz sweep, R da, res; W da on N^2 cells
            alg_bytes_per_launch = 3 * 8.0 * tile_cells / nl * (rf["aux"] / rf["count"])
        ach = alg_bytes_per_launch / (rf["ms"] / rf["count"] * 1e-3) / 1e9
        if sm == "rb":
            # dram__bytes_read.sum + dram__bytes_write.sum of one finest-level k_relax_rb launch (4 fused sweeps) at
            # 4096^2 x 4 from the ncu --set full capture profiles/ncu_r02/relax_rb.raw.csv (1.098 GB + 0.508 GB:
            # da and res read once with 128/112 halo redundancy, da written once, whatever the number of fused sweeps)
            traffic = 1.606e9 * tile_cells / (4096.0 * 4096 * 4) if nl == 4 else None
            kname = "k_relax_rb (finest level)"
            note = ("temporally blocked red-black sweeps: the fused sweeps of a launch are ONE pass over HBM, so the achieved rate "
                    "on pass-count algorithmic bytes may exceed the HBM peak; the kernel is bound by shared-memory bandwidth "
                    "and the fp64 pipe, not by DRAM")
        else:
            # profiles/ncu_r01/relax.raw.csv (1.143 GB + 0.559 GB; independent of the number of fused sweeps)
            traffic = 1.702e9 * tile_cells / (4096.0 * 4096 * 4) if nl == 4 else None
            kname = "k_relax_ws (finest level)"
            note = ("latency-bound wavefront (exact reference sweep order): the fused sweeps of a launch are ONE HBM pass, "
                    "so DRAM traffic is below the pass-count algorithmic bytes")
        roof = {"bound": "hbm", "kernel": kname, "achieved": ach, "peak": peak, "unit": "GB/s",
                "frac": ach / peak, "traffic": traffic, "peak_source": peak_src,
                "ms_per_launch": rf["ms"] / rf["count"], "sweeps_per_launch": rf["aux"] / rf["count"],
                "algorithmic_bytes_per_launch": alg_bytes_per_launch,
                "share_of_step": rf["ms"] / prof_ms_total if prof_ms_total > 0 else None, "note": note}
    kern_ms = {k: round(v["ms"] / psteps, 4) for k, v in prof.items()}
    # whole-step algorithmic bytes with the measured cycle counts (SURVEY.md 8(d))
    sweeps_all = prof["relax_fine"]["aux"] / psteps  # per step; every level does the same number of sweeps per cycle
    step_bytes = (2 * (ab["rhs"] + ab["residual"]) +
                  cycles / args.steps * (ab["restrict"] * 1.0 + ab["prolong"] * 1.0 + ab["correct"] + ab["residual"]) +
                  sweeps_all * ab["relax_sweep"] * 4.0 / 3) * cells
    step_roof = step_bytes / (ms_step * 1e-3) / 1e9
    # BASELINE metric, second half: wall-ms of one multigrid cycle (restriction of the residual, relax on every level,
    # prolongations, correction, residual) = the per-launch device times of those kernels over the timed region / cycles
    vcycle_ms = None
    if pcycles > 0:
        res = prof["residual"]
        vcycle_ms = (prof["relax_fine"]["ms"] + prof["relax_coarse"]["ms"] + prof["restrict"]["ms"] + prof["prolong"]["ms"] +
                     prof["correct"]["ms"] + (res["ms"] / res["count"] * pcycles if res["count"] else 0.)) / pcycles

    # ---- the other smoother on the same workload (1 GPU): the parity path (reference sweep order) next to the
    # throughput path; 3 timed steps after 2 warm-up, same event timing
    other = None
    if world == 1 and not args.no_other:
        osm = "lex" if sm == "rb" else "rb"
        try:
            m2 = G.Model(G.make_params(**workload_kw(N, nl)), local)
            m2.set_smoother(osm)
            m2.set_stream(stream.cuda_stream)
            m2.set(G.PSI, workload_psi(N, nl))
            m2.set_const()
            for _ in range(3):
                m2.step()
            c2 = m2.total_cycles
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(stream):
                f0.record(stream)
                for _ in range(3):
                    m2.step()
                f1.record(stream)
            f1.synchronize()
            oms = f0.elapsed_time(f1) / 3
            other = {"smoother": osm, "ms_per_step": oms, "value": cells / (oms * 1e-3), "unit": UNIT,
                     "mg_cycles_per_step": (m2.total_cycles - c2) / 3.0, "steps": 3}
            m2.close()
        except Exception as ex:
            other = {"smoother": osm, "error": repr(ex)}

    cpu = None
    if world == 1 and not args.no_cpu:
        try:
            # the reference-order OpenMP port on the FULL workload (same N, nl): 2 timed steps after 1 warm-up
            cv, cms, threads, _ = cpu_oracle_run(N, nl, 2, 1, "lex")
            cpu = {"value": cv, "unit": UNIT, "cores": threads, "kind": "port",
                   "sample": "the full %d^2 x nl=%d workload, 2 timed steps after 1 warm-up" % (N, nl),
                   "ms_per_step": cms}
        except Exception as ex:  # the baseline is a report, never a gate
            cpu = {"value": None, "unit": UNIT, "cores": 0, "kind": "port", "sample": "failed: %r" % (ex,)}

    this_mode = {"smoother": sm, "ms_per_step": ms_step, "value": value, "unit": UNIT, "roofline": roof,
                 "mg_cycles_per_step": cycles / args.steps}
    smoother_doc = ("rb = red-black ordering of the reference's relax_layer cell update (throughput mode; bit-exact against the "
                    "oracle with the same ordering, identical results on 1..8 GPUs; the reference documents its own sweep as "
                    "order/OpenMP/MPI dependent, poisson_layer.h:55-65); lex = the reference's serial sweep order (parity path)")
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64",
            "data": "synthetic",
            "config": {"workload": workload_name(N, nl), "N": N, "nl": nl, "smoother": sm, "smoothers": smoother_doc,
                       "parallelism": parallelism,
                       "l2": "inputs larger than L2 (each layer list is %.0f MB)" % (cells * 8 / 1e6),
                       "mg_cycles_per_step": cycles / args.steps},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": int(tile_cells * 8), "d2h_bytes_per_step": int(tile_cells * 8),
                    "steps": psteps_io, "ms_per_step": e2e_s / psteps_io * 1e3,
                    "mode": "pipelined: msqg_set_field_async / msqg_set_field_commit / msqg_get_field_async, double-buffered pinned host "
                            "buffers, uploads and downloads on their own streams beside the step",
                    "serial": {"value": e2e_serial_val, "ms_per_step": e2e_serial_s / esteps * 1e3, "steps": esteps,
                               "mode": "msqg_set_field; step; msqg_get_field"}},
            "roofline": roof, "cpu_baseline": cpu,
            ("fast_mode" if sm == "rb" else "parity_mode"): this_mode,
            ("parity_mode" if sm == "rb" else "fast_mode"): other,
            "kernel_ms_per_step": kern_ms, "vcycle_ms": vcycle_ms,
            "step_roofline": {"algorithmic_bytes_per_cell_layer_per_step": step_bytes / cells, "achieved": step_roof,
                              "peak": peak, "unit": "GB/s", "frac": step_roof / peak}}
    emit(line)
    if world > 1:
        m.close()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--N", type=int, default=N_DEFAULT)
    ap.add_argument("--nl", type=int, default=NL_DEFAULT)
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--no-other", action="store_true", help="skip the leg that times the other smoother (1 GPU)")
    ap.add_argument("--smoother", default="rb", choices=["rb", "lex"],
                    help="rb (default): red-black ordering of the relaxation sweep, the throughput mode, same result on any "
                         "number of GPUs; lex: the reference's serial sweep order (parity path; does not scale)")
    ap.add_argument("--modal", action="store_true",
                    help="vertical-mode inversion (MODE_PV_INVERT 1, eigmode.h; BASELINE config 3) instead of the layer-coupled solver")
    ap.add_argument("--periodic", action="store_true", help="datapoint: doubly periodic domain (sbc = -1)")
    ap.add_argument("--varRo", action="store_true", help="datapoint: Ro(y), i.e. horizontally varying stretching (with --modal: vertical modes)")
    ap.add_argument("--ensemble", action="store_true", help="BASELINE config 5: stochastic ensemble, --members per GPU of 512^2 x 3")
    ap.add_argument("--members", type=int, default=4)
    ap.add_argument("--ens-N", type=int, default=512, dest="ens_N")
    ap.add_argument("--noise", default="philox", choices=["philox", "libc"])
    ap.add_argument("--agg-n", type=int, default=0, dest="agg_n",
                    help="multi-GPU: levels with fewer than agg_n cells per side are not distributed (rb: replicated on every "
                         "GPU, default 512; lex: agglomerated on rank 0, default N)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None, dest="dump_outputs",
                    help="after the timed steps, write what the last one returned as DIR/{dt,t,psi,q}.npy (float64; "
                         "psi and q as a fixed seeded sample when larger than %d values)" % DUMP_SAMPLE)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "ours" and int(os.environ.get("WORLD_SIZE", "1")) > 1:
        ap.error("--dump-outputs supports the single-process run only")
    if args.agg_n <= 0:
        args.agg_n = args.N if args.smoother == "lex" else min(512, args.N)
    global MODAL, PERIODIC, VARRO
    MODAL = bool(args.modal)
    PERIODIC, VARRO = bool(args.periodic), bool(args.varRo)
    if PERIODIC:
        args.no_other = True   # the periodic domain runs with the red-black smoother only
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    elif args.ensemble:
        run_ensemble(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
