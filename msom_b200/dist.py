"""2-D domain decomposition of the msqg timestep (include/msqg.h layer 1b).

smoother="rb" (throughput mode): red-black sweeps are decomposition independent, so the group reproduces the
single-GPU red-black result bit for bit on any px x py; levels below `agg_n` are replicated on every GPU
(all-gather + redundant coarse solve) and each distributed level needs one deep-halo exchange per cycle.
smoother="lex" is the first-round decomposition of the reference-order sweep (block Gauss-Seidel, rank-0 coarse levels).

`Group(params, px, py, agg_n)` is the reference built with -D_MPI=1: px x py tiles, halo exchange
after every relaxation sweep, coarse levels below `agg_n` agglomerated on tile (0,0).

  * backend "local": all tiles in this process on one GPU (tests; emulates N ranks on one device)
  * backend "nccl" : one tile per process / GPU; torch.distributed only carries the 128-byte NCCL
    unique id to the other ranks (plumbing), the halo traffic is ncclSend/ncclRecv inside the library.
"""
import ctypes as C

import numpy as np

from . import capi as G

_bound = False


def _bind():
    global _bound
    L = G.lib()
    if _bound:
        return L
    vp, dp = C.c_void_p, np.ctypeslib.ndpointer(dtype=np.float64, flags="C_CONTIGUOUS")
    pd = C.POINTER(C.c_double)
    L.msqg_nccl_unique_id.argtypes = [C.c_char_p]
    L.msqg_group_create_local.argtypes = [C.POINTER(G.Params), C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
    L.msqg_group_create_nccl.argtypes = [C.POINTER(G.Params), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                         C.c_char_p, C.POINTER(vp)]
    L.msqg_group_create_local_sm.argtypes = [C.POINTER(G.Params), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.POINTER(vp)]
    L.msqg_group_create_nccl_sm.argtypes = [C.POINTER(G.Params), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int,
                                            C.c_char_p, C.POINTER(vp)]
    L.msqg_group_smoother.argtypes = [vp]
    L.msqg_group_transport.argtypes = [vp]
    L.msqg_group_destroy.argtypes = [vp]
    L.msqg_group_ntiles.argtypes = [vp]
    L.msqg_group_tile.argtypes = [vp, C.c_int]
    L.msqg_group_tile.restype = vp
    L.msqg_group_tile_info.argtypes = [vp, C.c_int, C.POINTER(C.c_int)]
    L.msqg_group_set_field.argtypes = [vp, C.c_int, C.c_int, dp]
    L.msqg_group_get_field.argtypes = [vp, C.c_int, C.c_int, dp]
    L.msqg_group_set_const.argtypes = [vp]
    L.msqg_group_invertq.argtypes = [vp, C.c_int]
    L.msqg_group_step.argtypes = [vp, C.c_double, C.c_double, pd, pd]
    L.msqg_group_last_mgstats.argtypes = [vp, C.POINTER(G.MgStats)]
    L.msqg_group_last_mode_mgstats.argtypes = [vp, C.c_int, C.POINTER(G.MgStats)]
    for f in ("msqg_group_total_cycles", "msqg_group_exchanges", "msqg_group_launches"):
        getattr(L, f).argtypes = [vp]
        getattr(L, f).restype = C.c_long
    L.msqg_group_set_stream_sync.argtypes = [vp]
    L.msqg_group_timer.argtypes = [vp, C.c_int, pd]
    L.msqg_group_profile_enable.argtypes = [vp, C.c_int]
    L.msqg_group_profile_read.argtypes = [vp, pd, C.POINTER(C.c_long), C.POINTER(C.c_long)]
    _bound = True
    return L


def grid_for(nranks):
    """process grid of SURVEY.md 8(e): 2x1, 2x2, 4x2 (px x py)"""
    return {1: (1, 1), 2: (2, 1), 4: (2, 2), 8: (4, 2)}[nranks]


def tile_box(N, px, py, rank):
    """(x0, y0, nx, ny) of rank = iy*px + ix on the finest level"""
    ix, iy = rank % px, rank // px
    nx, ny = N // px, N // py
    return ix * nx, iy * ny, nx, ny


class Group:
    def __init__(self, params, px, py, agg_n, device=0, backend="local", rank=0, nranks=1, uid=None, smoother="lex",
                 noise=None, seed=1):
        """noise, seed: the noise stream of a group with stochastic forcing (params.stochastic), required there:
        'philox' draws each tile's cells on the device (production), 'libc' replays the reference's rand() stream after
        srand(seed) on every tile (parity; each tile pays the host time of the whole N^2 nl stream per draw).  Every tile
        is seeded alike here; under NCCL every rank passes the same values."""
        self.L = _bind()
        if params.stochastic and noise not in ("libc", "philox"):
            raise G.MsqgError(G.ERR_ARG, "stochastic forcing on a group needs its noise stream: noise='philox' (device) or "
                                         "'libc' (host replay of the whole rand() stream on every tile), and the seed")
        self.p, self.px, self.py, self.agg_n = params, px, py, agg_n
        self.N, self.nl = params.N, params.nl
        h = C.c_void_p()
        sm = {"lex": 0, "rb": 1}[smoother]
        if backend == "local":
            G.check(self.L.msqg_group_create_local_sm(C.byref(params), device, px, py, agg_n, sm, C.byref(h)))
        else:
            G.check(self.L.msqg_group_create_nccl_sm(C.byref(params), device, px, py, agg_n, sm, rank, nranks, uid, C.byref(h)))
        self.smoother = smoother
        self.transport = "peer-memory" if self.L.msqg_group_transport(h) == 1 else "nccl"
        self.h = h
        self.t = 0.0
        self.ntiles = self.L.msqg_group_ntiles(self.h)
        self.boxes = []
        for t in range(self.ntiles):
            info = (C.c_int * 6)()
            self.L.msqg_group_tile_info(self.h, t, info)
            self.boxes.append(tuple(info))
        if params.stochastic:
            self.set_noise_mode(noise)
            self.seed_noise(seed)

    def close(self):
        if getattr(self, "h", None):
            self.L.msqg_group_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def nfields(self, fid):
        return self.L.msqg_nfields(self.L.msqg_group_tile(self.h, 0), fid)

    def set_tile(self, t, fid, arr):
        G.check(self.L.msqg_group_set_field(self.h, t, fid, np.ascontiguousarray(arr, dtype=np.float64)))

    def get_tile(self, t, fid):
        _, _, _, _, nx, ny = self.boxes[t]
        out = np.zeros((self.nfields(fid), ny, nx))
        G.check(self.L.msqg_group_get_field(self.h, t, fid, out))
        return out

    def set_global(self, fid, arr):
        """every local tile takes its block of the global [nf][N][N] array"""
        for t, (_, _, x0, y0, nx, ny) in enumerate(self.boxes):
            self.set_tile(t, fid, arr[:, y0:y0 + ny, x0:x0 + nx])

    def get_global(self, fid):
        """assemble the local tiles (all of them with the local backend) into a global array"""
        out = np.full((self.nfields(fid), self.N, self.N), np.nan)
        for t, (_, _, x0, y0, nx, ny) in enumerate(self.boxes):
            out[:, y0:y0 + ny, x0:x0 + nx] = self.get_tile(t, fid)
        return out

    def set_const(self):
        G.check(self.L.msqg_group_set_const(self.h))

    def _tiles(self):
        return [self.L.msqg_group_tile(self.h, t) for t in range(self.ntiles)]

    def seed_noise(self, seed):
        """stochastic forcing: seed the noise stream of every local tile like srand(seed) (libc mode) or as the Philox
        key (philox mode); the tiles then draw, each for its window, the field of the undecomposed model.  Under
        NCCL every rank calls this with the same seed (the group refuses to step otherwise)."""
        for h in self._tiles():
            self.L.msqg_seed_noise(h, seed)

    def set_noise_mode(self, mode):
        """'libc' replays the reference's rand() stream (every tile replays all N^2 nl draws, host time), 'philox'
        draws the field on the device (production).  Under NCCL every rank calls this with the same mode."""
        for h in self._tiles():
            G.check(self.L.msqg_set_noise_mode(h, {"libc": 0, "philox": 1}[mode]))

    def invertq(self, q_id=G.Q):
        G.check(self.L.msqg_group_invertq(self.h, q_id))

    def mgstats(self, mode=-1):
        """statistics of the last solve (mode < 0), or of vertical mode `mode` of the last modal inversion"""
        s = G.MgStats()
        G.check(self.L.msqg_group_last_mode_mgstats(self.h, mode, C.byref(s)))
        return s

    def step(self, tnext_event=-1.0):
        dt, tn = C.c_double(), C.c_double()
        G.check(self.L.msqg_group_step(self.h, self.t, tnext_event, C.byref(dt), C.byref(tn)))
        self.t = tn.value
        return dt.value

    def timer_start(self):
        G.check(self.L.msqg_group_timer(self.h, 0, None))

    def timer_stop(self):
        ms = C.c_double()
        G.check(self.L.msqg_group_timer(self.h, 1, C.byref(ms)))
        return ms.value

    def profile(self, on=True):
        G.check(self.L.msqg_group_profile_enable(self.h, 1 if on else 0))

    def profile_read(self):
        ms = (C.c_double * 9)(); cnt = (C.c_long * 9)(); aux = (C.c_long * 9)()
        G.check(self.L.msqg_group_profile_read(self.h, ms, cnt, aux))
        return {k: dict(ms=ms[i], count=cnt[i], aux=aux[i]) for i, k in enumerate(G.Model.PROF_CATS)}

    @property
    def total_cycles(self):
        return self.L.msqg_group_total_cycles(self.h)

    @property
    def exchanges(self):
        return self.L.msqg_group_exchanges(self.h)

    @property
    def launches(self):
        return self.L.msqg_group_launches(self.h)


def broadcast_bytes(payload, nbytes, device=None):
    """rank 0's `payload` (bytes of length nbytes) to every rank of the default process group"""
    import torch
    import torch.distributed as dist
    src = bytearray(payload if dist.get_rank() == 0 else bytes(nbytes))
    t = torch.frombuffer(src, dtype=torch.uint8).clone()
    if dist.get_backend() == "nccl":
        t = t.cuda(device)
    dist.broadcast(t, 0)
    return bytes(t.cpu().numpy().tobytes())


def nccl_group(params, agg_n, device, smoother="lex", noise=None, seed=1):
    """One tile per rank of the default torch.distributed process group (torch only carries the NCCL id).
    noise, seed: as Group (stochastic forcing), the same on every rank."""
    import torch.distributed as dist
    L = _bind()
    rank, world = dist.get_rank(), dist.get_world_size()
    px, py = grid_for(world)
    buf = C.create_string_buffer(128)
    if rank == 0:
        G.check(L.msqg_nccl_unique_id(buf))
    uid = broadcast_bytes(buf.raw, 128, device)
    return Group(params, px, py, agg_n, device, "nccl", rank, world, uid, smoother=smoother, noise=noise, seed=seed)
