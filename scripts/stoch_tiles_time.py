"""Cost of stochastic forcing on the tile machinery: deterministic steps against Philox-stochastic steps.

    python scripts/stoch_tiles_time.py [--steps 20] [--runs 3] [--out profiles/r05_stochastic_tiles.json]
        periodic 4096^2 x 4 on one GPU (the 1 x 1 periodic group behind msqg_create)
    torchrun --nproc-per-node 8 scripts/stoch_tiles_time.py --torchrun [--out ...]
        closed basin 8192^2 x 4, red-black, one tile per GPU (NCCL group, 4 x 2 tiles)

Each run builds a fresh model, warms up (recorded cycle graphs, first launches) and times `--steps` steps with a host
clock around work that ends in a device synchronise (every step synchronises for its dt).  The two variants alternate
(det, stoch, det, stoch, ...) so that other work on the host hits both alike; medians and spreads (max - min) are
reported.  A Philox draw reads sigma and writes the noise field once per step (2 x nl x N^2 doubles); the stochastic
right-hand side runs the L1-gather kernel k_rhs in place of the shared-memory k_rhs_t.  The JSON records the card name
and power limit read in the same process."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

STOCH = dict(stochastic=1, tr_stoch=10., amp_stoch=1.)


def card(index=0):
    r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    name, plim, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=plim, max_sm_clock=clk)


def summary(ms):
    return dict(median_ms_per_step=float(np.median(ms)), spread_ms=float(np.max(ms) - np.min(ms)), runs_ms_per_step=[float(x) for x in ms])


def time_runs(make, steps, warmup, runs):
    """alternating runs of the deterministic (False) and stochastic (True) variant; ms per step"""
    out = {False: [], True: []}
    for _ in range(runs):
        for stoch in (False, True):
            m, step, close = make(stoch)
            for _ in range(warmup):
                step()
            t0 = time.perf_counter()
            for _ in range(steps):
                step()
            out[stoch].append((time.perf_counter() - t0) * 1e3 / steps)
            close()
    return out


def periodic_one_gpu(args):
    import torch
    from common import base_kw, periodic_psi
    from msom_b200 import capi as G
    N, nl = 4096, 4
    psi = periodic_psi(N, nl)
    sig = np.full((nl, N, N), 1e-3) * (1 + np.arange(nl)[:, None, None])

    def make(stoch):
        m = G.Model(G.make_params(**base_kw(N, nl, sbc=-1., **(STOCH if stoch else {}))), 0)
        if stoch:
            m.L.msqg_seed_noise(m.h, 1234); G.check(m.L.msqg_set_noise_mode(m.h, 1))
            m.set(G.SSTOCH, sig)
        m.set(G.PSI, psi); m.set_const()
        return m, m.step, m.close

    r = time_runs(make, args.steps, args.warmup, args.runs)
    torch.cuda.synchronize()
    det, st = summary(r[False]), summary(r[True])
    return dict(workload="periodic %d^2 x %d, 1 GPU (1 x 1 periodic group, red-black), Philox noise" % (N, nl),
                card=card(0), steps_per_run=args.steps, warmup=args.warmup, runs=args.runs,
                deterministic=det, stochastic_philox=st,
                stochastic_over_deterministic=st["median_ms_per_step"] / det["median_ms_per_step"],
                noise_bytes_per_draw=2 * nl * N * N * 8)


def closed_basin_nccl(args):
    import torch
    import torch.distributed as dist
    from common import base_kw, synth_psi
    from msom_b200 import capi as G
    from msom_b200.dist import nccl_group
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    N, nl, agg_n = 8192, 4, 512
    psi = synth_psi(N, nl)
    sig = np.full((nl, N, N), 1e-3) * (1 + np.arange(nl)[:, None, None])

    def make(stoch):
        g = nccl_group(G.make_params(**base_kw(N, nl, **(STOCH if stoch else {}))), agg_n, local, smoother="rb",
                       noise="philox" if stoch else None, seed=1234)
        if stoch:
            g.set_global(G.SSTOCH, sig)
        g.set_global(G.PSI, psi); g.set_const()
        return g, g.step, g.close

    r = time_runs(make, args.steps, args.warmup, args.runs)
    det, st = summary(r[False]), summary(r[True])
    res = dict(workload="closed basin %d^2 x %d, %d GPUs (NCCL group, red-black, agg_n %d), Philox noise" % (N, nl, world, agg_n),
               card=card(local), steps_per_run=args.steps, warmup=args.warmup, runs=args.runs,
               deterministic=det, stochastic_philox=st,
               stochastic_over_deterministic=st["median_ms_per_step"] / det["median_ms_per_step"])
    dist.destroy_process_group()
    return res if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--torchrun", action="store_true", help="8192^2 x 4 closed basin, one tile per rank")
    ap.add_argument("--out", default=None, help="JSON file to merge the result into (key: periodic_1gpu / closed_basin_nccl)")
    args = ap.parse_args()
    res = closed_basin_nccl(args) if args.torchrun else periodic_one_gpu(args)
    if res is None:
        return
    print(json.dumps(res))
    if args.out:
        doc = json.load(open(args.out)) if os.path.exists(args.out) else {}
        doc["closed_basin_nccl" if args.torchrun else "periodic_1gpu"] = res
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
