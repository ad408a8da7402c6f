"""Randomised GPU-vs-oracle campaign for the per-vehicle local MIQP kernels (flat and cooperative).

    python scripts/stress_local.py [SEED] [--scale F]

SEED (default 0) seeds the draws; --scale F (default 1) multiplies every batch size, so that the campaign fits a test
budget (the oracle's time per problem grows ~4x per stage of horizon).  The kernel route follows the environment
(HVP_LOCAL_KERNEL, HVP_FLAT_STEAL, ...), read once per process.  Prints one line per case and `failures: K`."""
import argparse, os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np
import hybrid_vehicle_platoon_b200 as hvp
from oracle import oracle as O
from gen_cases import platoon_local_problems

ap = argparse.ArgumentParser()
ap.add_argument("seed", nargs="?", type=int, default=0)
ap.add_argument("--scale", type=float, default=1.0)
a = ap.parse_args()
rng = np.random.default_rng(a.seed)
bad = 0
for (N, n, S, stress, hetero, d0, t0) in ((6, 10, 2000, True, True, 10.0, 3.0), (6, 10, 2000, False, False, 50.0, 0.0),
                                          (4, 8, 1500, True, True, 50.0, 0.0), (8, 12, 300, True, True, 10.0, 3.0),
                                          (5, 6, 1500, True, False, 10.0, 3.0), (7, 10, 500, True, True, 50.0, 0.0),
                                          (9, 10, 100, True, True, 10.0, 3.0)):
    S = max(1, int(round(S * a.scale)))
    li = int(rng.integers(0, n))
    c = platoon_local_problems(rng, S, n, N, li, stress, hetero)
    args = (N, c["flags"], c["mass"], c["x0"], c["xf"], c["xb"], c["xl"])
    t = time.time()
    ro = O.local_miqp(*args, d0=d0, t0=t0)
    to = time.time() - t
    r = hvp.local_miqp(*args, d0=d0, t0=t0)
    ok = ro["status"] == 2
    st = (r["status"] == ro["status"]).mean()
    rel = np.abs(r["obj"][ok] - ro["obj"][ok]) / np.maximum(1.0, np.abs(ro["obj"][ok]))
    with np.errstate(invalid="ignore"):
        uniq = ok & ((ro["second"] - ro["obj"]) > 1e-6 * np.abs(ro["obj"]))
    du = np.abs(r["u"][uniq] - ro["u"][uniq]).max(initial=0.0)
    dm = (r["modes"][uniq] != ro["modes"][uniq]).any(axis=1).sum()
    flag = st < 1 or rel.max(initial=0.0) > 5e-7 or du > 1e-6 or dm > 0
    bad += int(flag)
    print(f"{'FAIL' if flag else 'ok  '} kernel={os.environ.get('HVP_LOCAL_KERNEL','auto')} steal={os.environ.get('HVP_FLAT_STEAL','1')} "
          f"N={N} n={n} B={S*n} li={li} stress={stress}: status_eq={st:.5f} opt={ok.mean():.3f} "
          f"uniq={uniq.mean():.3f} rel_obj_max={rel.max(initial=0.0):.2e} du_max={du:.2e} mode_mismatch={dm} nodes={r['nodes'].mean():.1f} (oracle {to:.1f}s)", flush=True)
print("failures:", bad)
sys.exit(1 if bad else 0)
