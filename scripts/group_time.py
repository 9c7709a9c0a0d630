"""python scripts/group_time.py [ROOT] : step time of local 2x2 groups (all four tiles on one GPU) with both smoothers,
timed with the group's CUDA events (msqg_group_timer).  ROOT is the tree whose library is loaded (default: this one), so
two builds can be compared in alternating processes.  One JSON line per configuration; `psi_sha` fingerprints the
state after the timed steps, so two trees that compute the same bits print the same value."""
import hashlib, json, os, subprocess, sys
ROOT = os.path.abspath(sys.argv[1]) if len(sys.argv) > 1 else os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from common import base_kw, synth_psi
from msom_b200 import capi as G
from msom_b200.dist import Group

WARMUP, STEPS = 3, 10
CONFIGS = [("lex", 1024, 4, 256), ("rb", 1024, 4, 256), ("rb", 2048, 4, 512)]   # smoother, N, nl, agg_n
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                     capture_output=True, text=True).stdout.strip()
for sm, N, nl, agg_n in CONFIGS:
    g = Group(G.make_params(**base_kw(N, nl)), 2, 2, agg_n, 0, smoother=sm)
    g.set_global(G.PSI, synth_psi(N, nl)); g.set_const()
    for _ in range(WARMUP):
        g.step()
    c0, x0 = g.total_cycles, g.exchanges
    g.timer_start()
    for _ in range(STEPS):
        g.step()
    ms = g.timer_stop()
    psi = g.get_global(G.PSI)
    print(json.dumps({"tree": os.path.basename(ROOT.rstrip("/")), "smoother": sm, "N": N, "nl": nl, "tiles": "2x2 local", "agg_n": agg_n,
                      "transport": g.transport, "ms_per_step": ms / STEPS, "cycles_per_step": (g.total_cycles - c0) / STEPS,
                      "exchanges_per_step": (g.exchanges - x0) / STEPS, "psi_sha": hashlib.sha256(psi.tobytes()).hexdigest()[:16],
                      "gpu": gpu}), flush=True)
    g.close()
