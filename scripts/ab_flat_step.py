"""A/B of two builds of libhvp.so on the bench step of the per-vehicle MIQP kernel (flat_miqp_kernel<6>).

    python scripts/ab_flat_step.py --old OLD_TREE [--new NEW_TREE] [--arm NAME=TREE ...] [--reps 5] [--steps 20]
                                   [--build-dir DIR] [--dump-dir DIR] [--scenarios 65536]

A TREE is a directory holding `hybrid_vehicle_platoon_b200/csrc` and `include`, e.g. an export of an older commit:

    mkdir -p /tmp/old && git archive HEAD~1 hybrid_vehicle_platoon_b200/csrc include | tar -x -C /tmp/old

`--new` defaults to this repository.  Every arm's sources are copied to `--build-dir/<name>` (default: a temporary
directory) and built there with the library's own Makefile, so the tree the script runs from is not written.  Each
arm's library is loaded by a worker process of its own, on bench.py's batch (make_batch(1234 + 1, S): 10 S problems),
and the workers are run in turn, `--reps` times each: one run = 3 warm-up steps and `--steps` timed steps, L2 flushed
(256 MiB write) between steps, each step timed by CUDA events.  The script then prints the median / min / max over the
runs of each arm's ms per step, with the card's name, power limit and maximum SM clock, and compares the solutions of
the first arm with every other arm: every status optimal, objectives equal to rtol 1e-9, inputs equal to 1e-7 wherever
the region sequences agree; a differing region sequence is accepted only between leaves whose objectives tie to 1e-9
(relative), because round-off may then pick either.  Exit status 1 when a comparison fails.
"""
import argparse
import json
import os
import shutil
import statistics
import subprocess
import sys
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
OUTPUTS = ("u", "x", "modes", "obj", "status")


def worker(lib_path, scenarios, dump_dir):
    """Loads `lib_path`, answers one timed run per line read from stdin with one JSON line."""
    sys.path.insert(0, ROOT)
    import torch
    from hybrid_vehicle_platoon_b200 import _lib
    _lib.LIB_PATH = lib_path                       # before the first lib() call
    import hybrid_vehicle_platoon_b200 as hvp
    from hybrid_vehicle_platoon_b200 import api
    from bench import HORIZON, N_VEH, make_batch
    dev = torch.device("cuda", 0)
    ctx = hvp.Context(0)
    batch = make_batch(1234 + 1, scenarios)
    B = scenarios * N_VEH
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).to(dev)
    ins = [t(batch[k]) for k in ("flags", "mass", "x0", "xf", "xb", "xl")]
    out = {"u": torch.empty((B, HORIZON), dtype=torch.float64, device=dev),
           "x": torch.empty((B, 2, HORIZON + 1), dtype=torch.float64, device=dev),
           "modes": torch.empty((B, HORIZON), dtype=torch.int32, device=dev),
           "obj": torch.empty(B, dtype=torch.float64, device=dev),
           "status": torch.empty(B, dtype=torch.int32, device=dev)}
    nodes = torch.empty(B, dtype=torch.int32, device=dev)
    iters = torch.empty(B, dtype=torch.int32, device=dev)
    desc = api.local_desc(HORIZON)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    stream = torch.cuda.current_stream().cuda_stream

    def step():
        api.local_miqp_device(desc, B, *ins, out["u"], out["x"], out["modes"], out["obj"], out["status"], nodes, iters,
                              ctx=ctx, stream=stream)

    first = True
    for line in sys.stdin:
        steps = int(line)
        for _ in range(3):
            step()
            flush.fill_(1)
        torch.cuda.synchronize()
        ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        for a, b in ev:
            a.record()
            step()
            b.record()
            flush.fill_(1)
        torch.cuda.synchronize()
        ms = [a.elapsed_time(b) for a, b in ev]
        if first:
            os.makedirs(dump_dir, exist_ok=True)
            for k, v in out.items():
                np.save(os.path.join(dump_dir, f"{k}.npy"), v.cpu().numpy())
            first = False
        print(json.dumps({"ms": ms, "nodes": float(nodes.double().mean()), "iters": float(iters.double().mean())}),
              flush=True)


def build(name, tree, build_root):
    dst = os.path.join(build_root, name)
    for sub in ("hybrid_vehicle_platoon_b200/csrc", "include"):
        shutil.copytree(os.path.join(tree, sub), os.path.join(dst, sub), dirs_exist_ok=True,
                        ignore=shutil.ignore_patterns("*.o", "*.so"))
    csrc = os.path.join(dst, "hybrid_vehicle_platoon_b200", "csrc")
    r = subprocess.run(["make", "-s", "-j", str(min(8, os.cpu_count() or 1)), "-C", csrc, "libhvp.so"],
                       capture_output=True, text=True)
    if r.returncode:
        sys.stderr.write(r.stdout[-3000:] + r.stderr[-3000:])
        raise SystemExit(f"building arm {name} from {tree} failed")
    return os.path.join(csrc, "libhvp.so")


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:                     # noqa: BLE001 -- reported, not fatal
        q = f"nvidia-smi unavailable ({e})"
    return q


def compare(ref_dir, dir_, name):
    a = {k: np.load(os.path.join(ref_dir, f"{k}.npy")) for k in OUTPUTS}
    b = {k: np.load(os.path.join(dir_, f"{k}.npy")) for k in OUTPUTS}
    ok = True
    not_opt = int((a["status"] != 2).sum() + (b["status"] != 2).sum())
    rel = np.abs(a["obj"] - b["obj"]) / np.maximum(np.abs(a["obj"]), 1e-300)
    same = (a["modes"] == b["modes"]).all(axis=1)
    du = float(np.abs(a["u"][same] - b["u"][same]).max()) if same.any() else 0.0
    dx = float(np.abs(a["x"][same] - b["x"][same]).max()) if same.any() else 0.0
    mism = np.nonzero(~same)[0]
    tie = rel[mism] <= 1e-9
    print(f"compare {name}: problems {len(same)}  non-optimal {not_opt}  obj max rel diff {rel.max():.2e}  "
          f"u max diff (same modes) {du:.2e}  x max diff (same modes) {dx:.2e}  mode mismatches {len(mism)} "
          f"(objective ties <= 1e-9: {int(tie.sum())})")
    if not_opt or not np.allclose(a["obj"], b["obj"], rtol=1e-9, atol=0) or du > 1e-7 or not tie.all():
        ok = False
        print(f"compare {name}: FAILED")
    return ok


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--old", help="tree of the old arm")
    ap.add_argument("--new", default=ROOT, help="tree of the new arm (default: this repository)")
    ap.add_argument("--arm", action="append", default=[], metavar="NAME=TREE", help="further arms")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--scenarios", type=int, default=65536)
    ap.add_argument("--build-dir", help="where the arms are built (default: a temporary directory)")
    ap.add_argument("--dump-dir", help="where each arm's outputs go as <arm>/<name>.npy (default: a temporary directory)")
    ap.add_argument("--worker", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.worker:
        worker(args.worker, args.scenarios, args.dump_dir)
        return
    arms = ([("old", args.old)] if args.old else []) + [("new", args.new)]
    for a in args.arm:
        name, tree = a.split("=", 1)
        arms.append((name, tree))
    if len(arms) < 2:
        ap.error("at least two arms are needed (--old TREE)")
    build_root = args.build_dir or tempfile.mkdtemp(prefix="ab_flat_build_")
    dump_root = args.dump_dir or tempfile.mkdtemp(prefix="ab_flat_out_")
    libs = {name: build(name, os.path.abspath(tree), build_root) for name, tree in arms}
    procs = {}
    for name, _ in arms:
        procs[name] = subprocess.Popen([sys.executable, os.path.abspath(__file__), "--worker", libs[name],
                                        "--scenarios", str(args.scenarios), "--dump-dir", os.path.join(dump_root, name)],
                                       stdin=subprocess.PIPE, stdout=subprocess.PIPE, text=True, cwd=ROOT)
    runs = {name: [] for name, _ in arms}
    info = {}
    try:
        for rep in range(args.reps):
            for name, _ in arms:
                p = procs[name]
                p.stdin.write(f"{args.steps}\n")
                p.stdin.flush()
                line = p.stdout.readline()
                if not line:
                    raise SystemExit(f"worker {name} died")
                r = json.loads(line)
                runs[name].append(float(np.mean(r["ms"])))
                info[name] = r
                print(f"rep {rep} {name}: {runs[name][-1]:.3f} ms/step (steps {min(r['ms']):.3f}-{max(r['ms']):.3f})",
                      flush=True)
    finally:
        for p in procs.values():
            p.stdin.close()
            p.wait()
    print(f"card: {card()}")
    B = args.scenarios * 10
    for name, _ in arms:
        v = runs[name]
        med = statistics.median(v)
        print(f"{name}: ms_per_step median {med:.3f} min {min(v):.3f} max {max(v):.3f} over {len(v)} runs of "
              f"{args.steps} steps; {B / (med * 1e-3) / 1e6:.2f} M solves/s; nodes/solve {info[name]['nodes']:.2f}, "
              f"qp iters/solve {info[name]['iters']:.2f}")
    ref = arms[0][0]
    ok = True
    for name, _ in arms[1:]:
        ok = compare(os.path.join(dump_root, ref), os.path.join(dump_root, name), f"{ref} vs {name}") and ok
    print(f"outputs: {dump_root}")
    sys.exit(0 if ok else 1)


if __name__ == "__main__":
    main()
