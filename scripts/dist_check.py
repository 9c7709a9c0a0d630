"""torchrun --nproc-per-node N scripts/dist_check.py [lex|rb|rbper|rbmodal|rbstoch|rbperstoch|rbvary] : the NCCL back-end of
the domain decomposition against the CPU oracle's emulation of the same decomposition, bit for bit, on every rank.
rbmodal: the vertical-mode inversion (mode_pv_invert = 1) on red-black tiles, every mode's statistics compared too.
rbstoch / rbperstoch: stochastic forcing with libc noise on the closed basin / the periodic domain: every rank replays
the reference's rand() stream from the same seed and keeps its tile's cells; the oracle draws from srand(seed).
rbvary: horizontally varying stretching, varRo > 0 together with a Fr(x, y) field (per-cell coefficient tables)."""
import os, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import torch, torch.distributed as dist
from common import base_kw, synth_psi
from oracle import oracle as O
from msom_b200 import capi as G
from msom_b200.dist import nccl_group, grid_for

rank, world, local = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"]), int(os.environ["LOCAL_RANK"])
torch.cuda.set_device(local)
dist.init_process_group("nccl", device_id=torch.device("cuda", local))
N, nl, agg_n = 256, 3, 64
sm = sys.argv[1] if len(sys.argv) > 1 else "lex"
modal = sm == "rbmodal"   # one scalar Helmholtz solve per vertical mode on the tiles
if modal:
    sm = "rb"
stoch = sm in ("rbstoch", "rbperstoch")
if stoch:
    sm = "rbper" if sm == "rbperstoch" else "rb"
STOCH = dict(stochastic=1, tr_stoch=10., amp_stoch=1.) if stoch else {}
vary = sm == "rbvary"
if vary:
    sm = "rb"
VARY = dict(varRo=1) if vary else {}
SEED = 2024
if sm == "rb":
    agg_n = 128 if world > 2 else 64
kw = base_kw(N, nl, mode_pv_invert=1) if modal else base_kw(N, nl, **STOCH, **VARY)
periodic = sm == "rbper"   # doubly periodic domain (sbc = -1) on the process grid: neighbours wrap around
if periodic:
    sm = "rb"
    kw = base_kw(N, nl, sbc=-1., **STOCH)
px, py = grid_for(world)
g = nccl_group(G.make_params(**kw), agg_n, local, smoother=sm, noise="libc" if stoch else None, seed=SEED)
psi = synth_psi(N, nl)
if periodic:
    from test_gpu_periodic import periodic_psi
    psi = periodic_psi(N, nl)
sig = np.full((nl, N, N), 1e-3) * (1 + np.arange(nl)[:, None, None])
if stoch:
    g.set_global(G.SSTOCH, sig)
fr = None
if vary:
    from test_gpu_dist_stretching import _fr_field
    fr = _fr_field(N, nl)
    g.set_global(G.FR, fr)
g.set_global(G.PSI, psi); g.set_const()
mo = O.Model(O.make_params(**kw)); mo.L.orc_set_decomp(mo.h, px, py, agg_n); mo.set_smoother(sm)
mo.set(O.PSI, psi)
if vary:
    mo.set(O.FR, fr)
if stoch:
    mo.set(O.SSTOCH, sig)
    import ctypes
    ctypes.CDLL(None).srand(SEED)
mo.set_const()
ok = not vary or g.stretching == "cells"
for s in range(3):
    ok &= (g.step() == mo.step())
if modal:
    for k in range(nl):
        sg, so = g.mgstats(k), mo.mgstats(k)
        ok &= (sg.i, sg.nrelax, sg.resb, sg.resa) == (so.i, so.nrelax, so.resb, so.resa)
_, _, x0, y0, nx, ny = g.boxes[0]
for fg, fo in ((G.PSI, O.PSI), (G.Q, O.Q)) + (((G.NSTOCH, O.NSTOCH),) if stoch else ()):
    ok &= bool(np.array_equal(g.get_tile(0, fg), mo.get(fo)[:, y0:y0 + ny, x0:x0 + nx]))
ok &= (g.total_cycles == mo.L.orc_total_cycles(mo.h))
t = torch.tensor([1 if ok else 0], device="cuda")
dist.all_reduce(t, op=dist.ReduceOp.MIN)
if rank == 0:
    print("DIST_CHECK", "PASS" if int(t.item()) == 1 else "FAIL", sm + ("-periodic" if periodic else "") + ("-modal" if modal else "") + ("-stochastic" if stoch else "") + ("-varying-stretching" if vary else ""), g.transport, "world", world, "grid %dx%d" % (px, py), "exchanges", g.exchanges)
g.close()
dist.destroy_process_group()
sys.exit(0 if int(t.item()) == 1 else 1)
