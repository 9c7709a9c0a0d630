"""Cost of horizontally varying stretching on tiles: group steps with uniform stretching, varRo (per-row tables) and a
Fr(x, y) field (per-cell tables).

    python scripts/stretch_tiles_time.py [--steps 20] [--runs 3] [--out profiles/r07_stretch_tiles.json]
        closed basin 4096^2 x 4 on ONE GPU as a local 2 x 2 group: an emulation of four tiles, not a scaling figure
    torchrun --nproc-per-node P scripts/stretch_tiles_time.py --torchrun [--out ...]
        closed basin 8192^2 x 4, red-black, one tile per GPU (NCCL group)

Each run builds a fresh group, warms up (recorded cycle graphs, first launches) and times `--steps` steps with a host
clock around work that ends in a device synchronise (every step synchronises for its dt).  The three variants alternate
(uniform, varRo, Fr(x, y), uniform, ...) so that other work on the host hits all alike; medians and spreads (max - min)
are reported.  The table memory per GPU is counted from the tile shapes: 6 nl doubles per row (varRo) or per cell
(Fr(x, y)) of every distributed level, halo margins included, plus the replicated coarse levels, per tile (one tile per
GPU under NCCL; the local emulation holds all four tiles on its GPU).  The JSON records the
card name and power limit read in the same process."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np  # noqa: E402

VARIANTS = ("uniform", "varRo", "frxy")


def card(index=0):
    r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    if r.returncode != 0:
        raise RuntimeError("nvidia-smi failed: " + r.stderr)
    name, plim, clk = [x.strip() for x in r.stdout.strip().splitlines()[0].split(",")]
    return dict(name=name, power_limit=plim, max_sm_clock=clk)


def summary(ms):
    return dict(median_ms_per_step=float(np.median(ms)), spread_ms=float(np.max(ms) - np.min(ms)), runs_ms_per_step=[float(x) for x in ms])


def fr_box(N, nl, Fr, x0, y0, nx, ny):
    """a smooth Fr(x, y) field (varies with x and y) on the cells [x0, x0 + nx) x [y0, y0 + ny)"""
    y, x = np.meshgrid((y0 + np.arange(ny) + 0.5) / N, (x0 + np.arange(nx) + 0.5) / N, indexing="ij")
    fr = np.zeros((nl, ny, nx))
    for l in range(nl - 1):
        fr[l] = Fr[l] * (1 + 0.3 * np.sin(2 * np.pi * x) * np.cos(np.pi * y))
    return fr


def table_bytes(N, nl, px, py, agg_n, per_cell):
    """stretching tables of one GPU: distributed levels (tile + halo margins of min(15, tile) cells on internal sides,
    counted on all four) and the replicated levels 1 .. below agg_n on the solver tile"""
    tot, n = 0, N
    while n >= 2:
        if n >= agg_n:
            tx, ty = n // px, n // py
            m = min(15, tx, ty)
            rows, cols = ty + 2 * m, tx + 2 * m
        else:
            rows, cols = n, n
        tot += (rows * cols if per_cell else rows) * 6 * nl * 8
        n //= 2
    return tot


def time_runs(make, steps, warmup, runs):
    out = {v: [] for v in VARIANTS}
    kinds = {}
    for _ in range(runs):
        for v in VARIANTS:
            g = make(v)
            kinds[v] = g.stretching
            for _ in range(warmup):
                g.step()
            t0 = time.perf_counter()
            for _ in range(steps):
                g.step()
            out[v].append((time.perf_counter() - t0) * 1e3 / steps)
            g.close()
    return out, kinds


def result(r, kinds, N, nl, px, py, agg_n, args, workload, crd):
    s = {v: summary(r[v]) for v in VARIANTS}
    return dict(workload=workload, card=crd, steps_per_run=args.steps, warmup=args.warmup, runs=args.runs,
                stretching_path=kinds, **s,
                varRo_over_uniform=s["varRo"]["median_ms_per_step"] / s["uniform"]["median_ms_per_step"],
                frxy_over_uniform=s["frxy"]["median_ms_per_step"] / s["uniform"]["median_ms_per_step"],
                table_bytes_per_tile=dict(varRo=table_bytes(N, nl, px, py, agg_n, False), frxy=table_bytes(N, nl, px, py, agg_n, True)))


def local_2x2(args):
    import torch
    from common import base_kw, synth_psi
    from msom_b200 import capi as G
    from msom_b200.dist import Group
    N, nl, px, py, agg_n = 4096, 4, 2, 2, 256
    psi = synth_psi(N, nl)
    fr = fr_box(N, nl, base_kw(N, nl)["Fr"], 0, 0, N, N)

    def make(v):
        g = Group(G.make_params(**base_kw(N, nl, **(dict(varRo=1) if v == "varRo" else {}))), px, py, agg_n, 0, smoother="rb")
        if v == "frxy":
            g.set_global(G.FR, fr)
        g.set_global(G.PSI, psi); g.set_const()
        return g

    r, kinds = time_runs(make, args.steps, args.warmup, args.runs)
    torch.cuda.synchronize()
    return result(r, kinds, N, nl, px, py, agg_n, args,
                  "closed basin %d^2 x %d, local %d x %d group on ONE GPU (emulation of the tiles, not a scaling figure), "
                  "red-black, agg_n %d" % (N, nl, px, py, agg_n), card(0))


def nccl(args):
    import torch
    import torch.distributed as dist
    from common import base_kw, synth_psi
    from msom_b200 import capi as G
    from msom_b200.dist import nccl_group, grid_for
    rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
    torch.cuda.set_device(local)
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    N, nl, agg_n = 8192, 4, 512
    px, py = grid_for(world)
    psi = synth_psi(N, nl)

    def make(v):
        g = nccl_group(G.make_params(**base_kw(N, nl, **(dict(varRo=1) if v == "varRo" else {}))), agg_n, local, smoother="rb")
        if v == "frxy":
            _, _, x0, y0, nx, ny = g.boxes[0]
            g.set_tile(0, G.FR, fr_box(N, nl, base_kw(N, nl)["Fr"], x0, y0, nx, ny))
        g.set_global(G.PSI, psi); g.set_const()
        return g

    r, kinds = time_runs(make, args.steps, args.warmup, args.runs)
    res = result(r, kinds, N, nl, px, py, agg_n, args,
                 "closed basin %d^2 x %d, %d GPUs (NCCL group %d x %d, red-black, agg_n %d)" % (N, nl, world, px, py, agg_n), card(local))
    dist.destroy_process_group()
    return res if rank == 0 else None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--torchrun", action="store_true", help="8192^2 x 4 closed basin, one tile per rank")
    ap.add_argument("--out", default=None, help="JSON file to merge the result into (key: local_2x2_1gpu / nccl_<P>gpu)")
    args = ap.parse_args()
    res = nccl(args) if args.torchrun else local_2x2(args)
    if res is None:
        return
    print(json.dumps(res))
    if args.out:
        key = "nccl_%dgpu" % int(os.environ["WORLD_SIZE"]) if args.torchrun else "local_2x2_1gpu"
        doc = json.load(open(args.out)) if os.path.exists(args.out) else {}
        doc[key] = res
        with open(args.out, "w") as f:
            json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
