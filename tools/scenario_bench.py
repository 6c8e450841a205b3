"""What evaluating L load scenarios costs: wva_analyze_scenarios against one full round per scenario, one GPU command.

For config 3 (1 000 x 8) and config 4 (10 000 x 8) and L in {1, 8, 64, 256} (scenario l scales every server's arrival
rate by a factor between 1/4 and 4, the same factors for both routes):
  (1) wva_analyze_scenarios: the decisions and per-type totals of all L scenarios copied back;
  (2) today's route, L times: wva_system_update_servers with the scenario's arrival rows, wva_analyze_pairs,
      wva_solve (unlimited) and wva_allocate_by_type, decisions and totals copied back.
Both are timed by CUDA events recorded on the context's stream around the whole route (every call of either route ends
in a stream synchronisation, so host work between the calls is inside the window); the two routes alternate within the
run.  Before the timed runs, one untimed pass of each route is compared byte for byte: every pair record and feasible
byte (wva_scenario_pairs_fetch against wva_pairs_fetch), every decision, count and cost.  Card name and power limit
are read in the same run.
    python tools/scenario_bench.py --runs 5 --out /tmp/scenarios/scenarios_cfg3_cfg4.json
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def _stats(xs):
    a = np.asarray(xs, dtype=np.float64)
    return dict(median=float(np.median(a)), min=float(a.min()), max=float(a.max()), n=int(len(a)))


def _card(dev):
    info = dict(name=torch.cuda.get_device_name(dev))
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(dev), "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["power_limit"], info["sm_max_clock"] = [x.strip() for x in q.split(",")]
    except Exception as e:                                   # the numbers are still reported, without the card's limits
        info["power_limit"] = "unavailable (%s)" % e
    return info


def _image(wva, k):
    if k == 3:
        return wva.synth.baseline_config(3)[0]
    c = wva.synth.CONFIGS[k]
    return wva.synth.make_system(c["S"], c["A"], seed=4, n_types=c["T"])


def _route_scenarios(ctx, rates):
    acc, _, cnt, cst = ctx.analyze_scenarios(rates)
    return acc, cnt, cst


def _route_rounds(ctx, base, rates, fetch=False):
    """L full rounds; returns (acc[L, S], count[L, T], cost[L, T], [(records, feasible)] if fetch)"""
    accs, cnts, csts, recs = [], [], [], []
    rows = base.shard(0, base.S)
    for l in range(rates.shape[0]):
        rows.srv_arrival_rpm[:] = rates[l]
        ctx.update_servers(0, rows)
        ctx.analyze_pairs(download=False)
        if fetch:
            recs.append(ctx.pairs_fetch())
        acc, _ = ctx.solve(unlimited=True)
        cnt, cst = ctx.allocate_by_type()
        accs.append(acc); cnts.append(cnt); csts.append(cst)
    return np.stack(accs), np.stack(cnts), np.stack(csts), recs


def run(wva, binding, k, L, runs, warmup):
    base = _image(wva, k)
    rates = (base.srv_arrival_rpm.astype(np.float64)[None, :] *
             np.geomspace(0.25, 4.0, L)[:, None] if L > 1 else base.srv_arrival_rpm[None, :].astype(np.float64)).astype(np.float32)
    ctx = binding.Context(0)
    try:
        ctx.upload(base.shard(0, base.S))
        stream = torch.cuda.ExternalStream(ctx.stream(), device=torch.device("cuda", 0))
        # byte-for-byte check of the two routes
        s_acc, s_cnt, s_cst = _route_scenarios(ctx, rates)
        s_recs = [ctx.scenario_pairs_fetch(l) for l in range(L)]
        r_acc, r_cnt, r_cst, r_recs = _route_rounds(ctx, base, rates, fetch=True)
        same = bool(np.array_equal(s_acc, r_acc) and np.array_equal(s_cnt, r_cnt) and s_cst.tobytes() == r_cst.tobytes())
        for (a, fa), (b, fb) in zip(s_recs, r_recs):
            same = same and bool(np.array_equal(fa, fb)) and a.equal_bits(b)[0]
        feasible = int(sum(int(f.sum()) for _, f in s_recs))
        times = dict(scenarios=[], rounds=[])
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for i in range(warmup + runs):
            for route in ("scenarios", "rounds") if i % 2 == 0 else ("rounds", "scenarios"):
                e0.record(stream)
                if route == "scenarios":
                    _route_scenarios(ctx, rates)
                else:
                    _route_rounds(ctx, base, rates)
                e1.record(stream)
                e1.synchronize()
                if i >= warmup:
                    times[route].append(e0.elapsed_time(e1))
        phase_us = ctx.phase_usec(wva.abi.PHASE_SCENARIOS)
        med1, med2 = np.median(times["scenarios"]), np.median(times["rounds"])
        return dict(config=k, servers=base.S, accelerators=base.A, scenarios=L, feasible_records=feasible,
                    same_bytes_both_routes=same, analyze_scenarios_ms=_stats(times["scenarios"]),
                    rounds_ms=_stats(times["rounds"]), speedup_median=float(med2 / med1),
                    last_phase_scenarios_us=int(phase_us))
    finally:
        ctx.close()


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--runs", type=int, default=5, help="timed runs of each route per (config, L)")
    ap.add_argument("--warmup", type=int, default=1)
    ap.add_argument("--configs", default="3,4")
    ap.add_argument("--scenarios", default="1,8,64,256")
    ap.add_argument("--out", default=None, help="JSON output path")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("scenario_bench.py measures on a GPU; none is visible")
    import wva_import
    wva = wva_import.load()
    from inferno_autoscaler_b200 import binding
    res = dict(card=_card(0), method="CUDA events on the context's stream around each whole route; the routes alternate "
                                      "within the run; results of both routes compared byte for byte before timing")
    res["runs"] = [run(wva, binding, int(k), int(L), args.runs, args.warmup)
                   for k in args.configs.split(",") for L in args.scenarios.split(",")]
    text = json.dumps(res, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
