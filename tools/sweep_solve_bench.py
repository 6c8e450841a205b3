"""What solving over the sweep's per-pair winners costs and buys (one GPU command).

  (a) config 3: the sweep phase (WVA_PHASE_GRID) of bench.py's step with per-pair winners off and on,
      alternating within the run;
  (b) config 4 with capacities at 60 % of the unconstrained pair-record demand (as `bench.py --limited` sets
      them): analyze + limited solve (PriorityExhaustive) + totals, over the pair records (wva_solve) and over
      the sweep records (wva_solve_grid), alternating: step time, solve phase, servers allocated, per-type
      counts and summed cost;
  (c) the same as (b) on 2 GPUs through wva_comm_* (one process per GPU), when the box has them.

CUDA events on the library's stream; L2 flushed (256 MB write) before every timed step, as bench.py does.
Writes the JSON to --out and prints it.
    python tools/sweep_solve_bench.py --steps 20 --out /tmp/sweep_solve_bench.json
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


class Timer:
    def __init__(self, ctx, dev):
        self.stream = torch.cuda.ExternalStream(ctx.stream(), device=dev)
        self.flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)
        self.i = 0

    def __call__(self, f):
        """device ms of f() on the library's stream, L2 flushed before"""
        self.i += 1
        self.flush.fill_(self.i & 0xff)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(self.stream)
        f()
        e1.record(self.stream)
        torch.cuda.synchronize()
        return e0.elapsed_time(e1)


def part_a(wva, binding, steps, warmup):
    img, c = wva.synth.baseline_config(3)
    R, B = c["r_max"], c["b_max"]
    ctx = binding.Context(0)
    try:
        ctx.upload(img)
        tm = Timer(ctx, torch.device("cuda", 0))
        want_cube = True                                    # bench.py's default step at config 3 materialises the cube
        for _ in range(warmup):
            for on in (False, True):
                ctx.grid_set_pair_winners(on)
                ctx.analyze(R, B, want_cube=want_cube)
        res = {False: dict(step_ms=[], grid_us=[], launches=[]), True: dict(step_ms=[], grid_us=[], launches=[])}
        for i in range(2 * steps):
            on = bool(i & 1)
            ctx.grid_set_pair_winners(on)
            n0 = ctx.launch_count()
            ms = tm(lambda: ctx.analyze(R, B, want_cube=want_cube))
            res[on]["step_ms"].append(ms)
            res[on]["grid_us"].append(ctx.phase_usec(wva.abi.PHASE_GRID))
            res[on]["launches"].append(ctx.launch_count() - n0)
        out = {}
        for on, r in res.items():
            out["pair_winners_" + ("on" if on else "off")] = dict(analyze_ms=_stats(r["step_ms"]), grid_phase_us=_stats(r["grid_us"]),
                                                                  launches=sorted(set(r["launches"])))
        off, on_ = out["pair_winners_off"]["grid_phase_us"]["median"], out["pair_winners_on"]["grid_phase_us"]["median"]
        out["grid_phase_delta_pct"] = 100.0 * (on_ - off) / off
        return dict(config=3, servers=img.S, accelerators=img.A, r_max=R, b_max=B, **out)
    finally:
        ctx.close()


def limited_image(wva, binding, dev):
    """config 4, capacities at 60 % of the unconstrained pair-record demand (bench.py --limited)"""
    c = wva.synth.CONFIGS[4]
    img = wva.synth.make_system(c["S"], c["A"], seed=4, n_types=c["T"])
    ctx = binding.Context(dev)
    try:
        ctx.upload(img)
        ctx.analyze_pairs(download=False)
        _, ch0 = ctx.solve(unlimited=True)
        wva.synth.set_capacity_from_demand(img, ch0.acc, ch0.num_replicas, fraction=0.6)
    finally:
        ctx.close()
    return img, c


def limited_steps(wva, ctx, img, c, tm, steps, warmup, comm=False):
    """analyze + limited solve + totals over each record set, alternating"""
    R, B = c["r_max"], c["b_max"]
    pol = wva.abi.POLICY_PRIORITY_EXHAUSTIVE
    ctx.grid_set_pair_winners(True)
    want_cube = False                                        # 10 000 servers: 1.3 G candidates, no cube (bench.py --no-cube size)

    def place():
        ctx.upload(img)
        if comm:
            ctx.comm_shard()

    def step(src):
        ctx.analyze(R, B, want_cube=want_cube)
        (ctx.solve_grid if src == "sweep" else ctx.solve)(unlimited=False, policy=pol, download=False)
        ctx.allocate_by_type(download=False)

    place()
    for _ in range(warmup):
        for src in ("pairs", "sweep"):
            step(src)
    res = {s: dict(step_ms=[], solve_us=[]) for s in ("pairs", "sweep")}
    for i in range(2 * steps):
        src = ("pairs", "sweep")[i & 1]
        res[src]["step_ms"].append(tm(lambda: step(src)))
        res[src]["solve_us"].append(ctx.phase_usec(wva.abi.PHASE_SOLVE))
    out = {}
    for src in ("pairs", "sweep"):
        ctx.analyze(R, B)
        acc, chosen = (ctx.solve_grid if src == "sweep" else ctx.solve)(unlimited=False, policy=pol)
        cnt, cst = ctx.allocate_by_type()
        out[src] = dict(step_ms=_stats(res[src]["step_ms"]), solve_phase_us=_stats(res[src]["solve_us"]),
                        servers_allocated=int((acc >= 0).sum()), type_counts=[int(x) for x in cnt],
                        type_costs=[float(x) for x in cst], total_cost=float(np.sum(cst.astype(np.float64))))
    out["capacity"] = [int(x) for x in img.type_capacity]
    return out


def part_b(wva, binding, steps, warmup):
    img, c = limited_image(wva, binding, 0)
    ctx = binding.Context(0)
    try:
        tm = Timer(ctx, torch.device("cuda", 0))
        return dict(config=4, servers=img.S, accelerators=img.A, policy="PriorityExhaustive",
                    **limited_steps(wva, ctx, img, c, tm, steps, warmup))
    finally:
        ctx.close()


def _rank(rank, world, port, steps, warmup, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    import wva_import
    wva = wva_import.load()
    from inferno_autoscaler_b200 import binding, distributed as D
    img, c = limited_image(wva, binding, rank)
    ctx = binding.Context(rank)
    D.attach_library_comm(ctx, dev)
    tm = Timer(ctx, dev)
    out = limited_steps(wva, ctx, img, c, tm, steps, warmup, comm=True)
    q.put((rank, out))
    ctx.comm_destroy()
    ctx.close()
    dist.destroy_process_group()


def part_c(steps, warmup):
    if torch.cuda.device_count() < 2:
        return dict(skipped="the box has %d GPU" % torch.cuda.device_count())
    import torch.multiprocessing as mp
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    port = 29900 + (os.getpid() % 1000)
    procs = [mpc.Process(target=_rank, args=(r, 2, port, steps, warmup, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=1800) for _ in procs)
    for p in procs:
        p.join(timeout=120)
    return dict(config=4, gpus=2, policy="PriorityExhaustive", rank0=res[0], rank1=res[1])


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--steps", type=int, default=20, help="timed steps per variant")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", default=None, help="JSON output path")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be >= 1")
    if not torch.cuda.is_available():
        sys.exit("sweep_solve_bench: no CUDA device")
    import __graft_entry__ as ge
    ge.build_cuda()
    import wva_import
    wva = wva_import.load()
    from inferno_autoscaler_b200 import binding
    rep = dict(card=_card(0), gpus=torch.cuda.device_count(), steps=args.steps, warmup=args.warmup,
               timing="CUDA events on the library stream; L2 flushed (256 MB write) before every timed step")
    rep["a_sweep_overhead"] = part_a(wva, binding, args.steps, args.warmup)
    rep["b_limited_one_gpu"] = part_b(wva, binding, args.steps, args.warmup)
    rep["c_limited_two_gpus"] = part_c(args.steps, args.warmup)
    text = json.dumps(rep, indent=1)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(text + "\n")
    print(text)


if __name__ == "__main__":
    main()
