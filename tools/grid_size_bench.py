"""What sizing the sweep's per-pair records costs (wva_grid_pairs_size), one GPU command.

For config 3 (1 000 x 8) and config 4 (10 000 x 8) on one GPU: the sweep with per-pair winners on, then
  (new)  wva_grid_pairs_size: device time of WVA_PHASE_GRID_SIZE, and wall time of the call;
  (old)  the long way round for the same records: wva_grid_pairs_fetch, one wva_queue_config + target row per record
         built on the host, wva_queue_size (one thread per request), the rates written back -- wall time, copies included.
The two alternate within the run, each on records fresh from a sweep; the status histogram and the number of records
are reported, and both ways are checked to give the same rates.  Then bench.py (default config) runs in the same
command, for the pairs and sweep phases.  Card name and power limit are read in the same run.
    python tools/grid_size_bench.py --runs 30 --out /tmp/grid_size/grid_size_cfg3_cfg4.json
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def _stats(xs):
    a = np.asarray(xs, dtype=np.float64)
    return dict(median=float(np.median(a)), min=float(a.min()), max=float(a.max()),
                p25=float(np.percentile(a, 25)), p75=float(np.percentile(a, 75)), n=int(len(a)))


def _card(dev):
    info = dict(name=torch.cuda.get_device_name(dev))
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:                                   # the numbers are still reported, without the card's limits
        info["power_limit"] = "unavailable (%s)" % e
    return info


def _old_way(wva, ref, ctx, img):
    """fetch, host-built configs, wva_queue_size: (sized max_arrv of the records, status)"""
    recs, fe = ctx.grid_pairs_fetch()
    gi, cfgs, targets = ref.size_inputs(wva, img, fe)
    b = recs.batch_size[gi]
    cfgs["max_batch_size"] = b
    cfgs["max_queue_size"] = b * wva.abi.MAX_QUEUE_TO_BATCH_RATIO
    _, m, _, st = ctx.queue_size(cfgs, targets)
    ok = st == 0
    rate = recs.max_arrv_rate_per_replica.copy()
    rate[gi[ok]] = (m["throughput"][ok] / np.float32(1000)).astype(np.float32)
    status = np.zeros(len(fe), dtype=np.uint8)
    status[gi] = np.where(ok, 1, 2)
    return rate, status


def run_config(wva, binding, ref, k, runs, warmup):
    c = dict(wva.synth.CONFIGS[k])
    img = wva.synth.baseline_config(3)[0] if k == 3 else wva.synth.make_system(c["S"], c["A"], seed=4, n_types=c["T"])
    R, B = c["r_max"], c["b_max"]
    ctx = binding.Context(0)
    try:
        ctx.upload(img)
        ctx.grid_set_pair_winners(True)
        new_us, new_wall, old_wall = [], [], []
        hist = n_rec = None
        for i in range(warmup + runs):
            for way in ("new", "old") if i % 2 == 0 else ("old", "new"):
                ctx.analyze_grid_device(R, B)
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                if way == "new":
                    status = ctx.grid_pairs_size()
                else:
                    o_rate, o_status = _old_way(wva, ref, ctx, img)
                dt = (time.perf_counter() - t0) * 1e3
                if i < warmup:
                    continue
                if way == "new":
                    new_wall.append(dt)
                    new_us.append(ctx.phase_usec(wva.abi.PHASE_GRID_SIZE))
                    n_rec = int((status > 0).sum())
                    hist = np.bincount(status, minlength=3).tolist()
                    n_rate = ctx.grid_pairs_fetch()[0].max_arrv_rate_per_replica
                else:
                    old_wall.append(dt)
        same = bool(np.array_equal(o_status, status) and np.array_equal(o_rate.view(np.uint32), n_rate.view(np.uint32)))
        return dict(config=k, servers=img.S, accelerators=img.A, r_max=R, b_max=B, records=n_rec,
                    status_histogram=dict(no_record=hist[0], sized=hist[1], size_error=hist[2]),
                    grid_pairs_size_device_us=_stats(new_us), grid_pairs_size_wall_ms=_stats(new_wall),
                    fetch_queue_size_wall_ms=_stats(old_wall), same_rates_both_ways=same)
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--runs", type=int, default=30, help="timed runs of each way per config (>= 20)")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--out", default=None, help="JSON output path")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("grid_size_bench.py measures on a GPU; none is visible")
    import wva_import
    wva = wva_import.load()
    from inferno_autoscaler_b200 import binding
    import grid_size_ref as ref
    res = dict(card=_card(0), method="CUDA events of WVA_PHASE_GRID_SIZE (device time of the call); wall times by the host clock "
                                        "around calls that end in a device synchronisation; the two ways alternate within the run")
    res["configs"] = [run_config(wva, binding, ref, k, args.runs, args.warmup) for k in (3, 4)]
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "20", "--warmup", "3"],
                       capture_output=True, text=True, cwd=ROOT)
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    res["bench_py_default"] = json.loads(lines[-1]) if lines else dict(rc=p.returncode, stderr=p.stderr[-2000:])
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
