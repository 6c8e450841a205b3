"""GPU: the candidate sweep's per-(server, accelerator) winners as solver input (wva_grid_set_pair_winners,
wva_grid_pairs_fetch, wva_solve_grid), against the oracle.

  1. config 2, exhaustive: records + feasible bytes equal the oracle's in every sweep mode;
  2. the option changes none of the sweep's other outputs (stop-and-go and fused flows) nor its launch count;
  3. config 3 and 4 slices: every record proved (own candidate re-evaluated, no feasible candidate with a smaller
     (value, r, b) in its pair, no feasible candidate at all in a pair flagged infeasible);
  4. unlimited / limited solves over the records (every policy, delayed best-effort, all three greedy paths);
  5. the records' lifetime (WVA_ESTATE cases), with the pair-record solve unaffected;
  6. two GPUs: the in-library exchange and wva_group."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import sweep_pair_ref as ref

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32
MAX_F32 = np.finfo(np.float32).max
FIELDS = ("acc", "num_replicas", "batch_size", "cost", "value", "itl", "ttft", "rho", "max_arrv_rate_per_replica")


def _threads(oracle):
    return max(1, oracle.hardware_threads())


def _reset(ctx, img=None):
    ctx.grid_set_pair_winners(False)
    ctx.set_certified_tails(1)
    ctx.grid_set_fused(True)
    ctx.solve_set_ranked(2)
    if img is not None:
        ctx.set_shard(0, img.S)


def _records_equal(a, b):
    ok, field = a.equal_bits(b)
    assert ok, field


def test_config2_records_equal_oracle_in_every_mode(wva, oracle, ctx):
    img, c = wva.synth.baseline_config(2)
    R, B = c["r_max"], c["b_max"]
    o_best, o_cube, o_status, _ = oracle.analyze_grid(img, R, B, want_cube=True, threads=_threads(oracle))
    want, wfe = ref.pair_records(wva, oracle, img, R, B, o_cube, o_status)
    assert 0 < int(wfe.sum()) < img.S * img.A
    try:
        ctx.upload(img)
        ctx.grid_set_pair_winners(True)
        for mode in (1, 0, 3, 5, 9, 17):
            ctx.set_certified_tails(mode)
            best, _, _ = ctx.analyze_grid(R, B)
            assert best.tobytes() == o_best.tobytes(), mode
            got, gfe = ctx.grid_pairs_fetch()
            assert np.array_equal(gfe, wfe), mode
            _records_equal(got, want)
    finally:
        _reset(ctx)


def test_option_changes_no_other_output(wva, ctx):
    """500 servers of config 3 (as test_config3_fused_sweep_vs_oracle): winners, cube and status are the same bytes
    with the option on and off, in the stop-and-go and the fused flow, and the sweep launches as many kernels."""
    img, c = wva.synth.baseline_config(3)
    R, B = c["r_max"], c["b_max"]
    import hashlib
    try:
        ctx.upload(img)
        ctx.set_shard(250, 500)
        for fused in (False, True):
            ctx.grid_set_fused(fused)
            seen = []
            for on in (False, True, False):
                ctx.grid_set_pair_winners(on)
                n0 = ctx.launch_count()
                best, cube, status = ctx.analyze_grid(R, B, want_cube=True)
                seen.append((best.tobytes(), hashlib.sha256(cube.data).digest(), hashlib.sha256(status.data).digest(),
                             ctx.launch_count() - n0, ctx.grid_last_fused()))
                del cube, status
            assert seen[0] == seen[1] == seen[2], fused
            assert seen[1][4] == (1 if fused else 0)
    finally:
        _reset(ctx, img)


def _prove_records(wva, oracle, ctx, img, first, count, R, B):
    """Sweep servers [first, first+count) with the option on and prove every pair record against the oracle."""
    th = _threads(oracle)
    A = img.A
    ctx.upload(img)
    ctx.set_shard(first, count)
    ctx.grid_set_pair_winners(True)
    best, _, _ = ctx.analyze_grid(R, B)
    got, gfe = ctx.grid_pairs_fetch()
    lo, hi = first * A, (first + count) * A
    assert (gfe[:lo] == 0).all() and (gfe[hi:] == 0).all() and (got.acc[:lo] == 0).all() and (got.acc[hi:] == 0).all()
    fe = gfe[lo:hi].reshape(count, A).astype(bool)
    sl, a = np.nonzero(fe)
    gi = (sl + first) * A + a
    r = got.num_replicas[gi].astype(np.int32)
    b = got.batch_size[gi].astype(np.int32)
    assert np.array_equal(got.acc[gi], a)
    # (1) each record is its own candidate, re-evaluated by the oracle
    m, st = oracle.grid_candidates(img, sl + first, a, r, b, threads=th)
    assert (st == (wva.abi.CAND_OK | wva.abi.CAND_FEASIBLE)).all()
    vals = oracle.grid_row_values(img, R, first, first + count)          # [count, A, R]
    want = ref.candidate_fields(img, sl + first, a, r, b, vals[sl, a, r - 1], m)
    for name in FIELDS:
        g = getattr(got, name)[gi]
        w = want[name]
        if g.dtype == np.float32:
            g, w = g.view(np.uint32), w.view(np.uint32)
        assert np.array_equal(g, w), name
    # infeasible pairs of the shard hold the empty record
    off = np.flatnonzero(~fe.reshape(-1)) + lo
    assert (got.acc[off] == ref.ACC_NONE).all() and (got.num_replicas[off] == 0).all()
    # (2) no feasible candidate with a smaller (value, r, b) in the same pair, (3) none at all in an infeasible pair
    r_ix = np.arange(1, R + 1)[None, None, :]
    v_win = np.full((count, A), np.inf, dtype=F)
    r_win = np.full((count, A), R + 1)
    v_win[sl, a] = got.value[gi]
    r_win[sl, a] = r
    with np.errstate(invalid="ignore"):
        lower = (vals < v_win[..., None]) | ((vals == v_win[..., None]) & (r_ix < r_win[..., None]))   # NaN rows: never selected
    ls, la, lr = np.nonzero(lower)
    rows_s = np.concatenate([ls, sl]).astype(np.int32) + first
    rows_a = np.concatenate([la, a]).astype(np.int32)
    rows_r = np.concatenate([lr + 1, r]).astype(np.int32)
    b_lo = np.ones(len(rows_s), dtype=np.int32)
    b_hi = np.concatenate([np.full(len(ls), B), b - 1]).astype(np.int32)
    nf = oracle.grid_rows_feasible(img, rows_s, rows_a, rows_r, b_lo, b_hi, threads=th)
    assert int(nf.sum()) == 0, "the oracle finds a feasible candidate that precedes a pair record"
    # the server winners are the best of their pairs' records
    acc, rep, bat, _ = ref.best_of_pairs(got, gfe, img.S, A)
    acc, rep, bat = acc[first:first + count], rep[first:first + count], bat[first:first + count]
    assert np.array_equal(acc, best["acc"])
    has = acc >= 0
    assert np.array_equal(rep[has], best["replicas"][has]) and np.array_equal(bat[has], best["batch"][has])
    return dict(pairs=count * A, feasible_pairs=len(gi), proof_candidates=int((b_hi - b_lo + 1).clip(min=0).sum()))


def test_config3_and_config4_slices_records_proved(wva, oracle, ctx):
    tot = dict(pairs=0, feasible_pairs=0, proof_candidates=0)
    try:
        img, c = wva.synth.baseline_config(3)
        for first in (0, 500):
            rep = _prove_records(wva, oracle, ctx, img, first, 32, c["r_max"], c["b_max"])
            for k in tot:
                tot[k] += rep[k]
        c = wva.synth.CONFIGS[4]
        img = wva.synth.make_system(c["S"], c["A"], seed=4, n_types=c["T"])
        for first in (0, 9968):
            rep = _prove_records(wva, oracle, ctx, img, first, 32, c["r_max"], c["b_max"])
            for k in tot:
                tot[k] += rep[k]
    finally:
        _reset(ctx, img)
    assert tot["feasible_pairs"] > 100
    print("per-pair records proved:", tot)


def test_unlimited_solve_grid_picks_sweep_winners(wva, oracle, ctx):
    img, c = wva.synth.baseline_config(3)
    try:
        ctx.upload(img)
        ctx.grid_set_pair_winners(True)
        ctx.analyze(c["r_max"], c["b_max"])
        best = ctx.grid_fetch()
        acc, chosen = ctx.solve_grid(unlimited=True)
        win = (best["acc"] >= 0) & (best["value"] < MAX_F32)
        assert win.sum() > 300
        assert np.array_equal(acc[win], best["acc"][win]) and (acc[~win] == -1).all()
        assert np.array_equal(chosen.num_replicas[win], best["replicas"][win].astype(np.int64))
        assert np.array_equal(chosen.batch_size[win], best["batch"][win].astype(np.int64))
        assert np.array_equal(chosen.cost[win].view(np.uint32), best["cost"][win].view(np.uint32))
        cnt, cst = ctx.allocate_by_type()
        w_cnt, w_cst = oracle.allocate_by_type(img, acc, chosen)
        assert np.array_equal(cnt, w_cnt) and cst.tobytes() == w_cst.tobytes()
        # unlimited does not consume the records; the pair-record solve still runs on its own records
        ctx.grid_pairs_fetch()
        p_acc, _ = ctx.solve(unlimited=True)
        o_pairs, o_feas, _ = oracle.analyze_pairs(img, threads=_threads(oracle))
        w_acc, _ = oracle.solve(img, o_pairs, o_feas, unlimited=True)
        assert np.array_equal(p_acc, w_acc)
    finally:
        _reset(ctx, img)


def test_limited_solve_grid_vs_oracle_every_policy_and_path(wva, oracle, ctx):
    """config 4 (10 000 x 8) with caps at 60 % of the sweep records' own unlimited demand"""
    c = wva.synth.CONFIGS[4]
    img = wva.synth.make_system(c["S"], c["A"], seed=4, n_types=c["T"])
    R, B = c["r_max"], c["b_max"]
    A = wva.abi
    from inferno_autoscaler_b200.binding import WvaError
    try:
        ctx.upload(img)
        ctx.grid_set_pair_winners(True)
        ctx.analyze_grid_device(R, B)
        recs, feas = ctx.grid_pairs_fetch()
        u_acc, u_chosen = ctx.solve_grid(unlimited=True)
        demand = wva.synth.set_capacity_from_demand(img, u_acc, u_chosen.num_replicas, fraction=0.6)
        assert (demand > img.type_capacity).any()                   # the caps bind
        ctx.set_capacity(img.type_capacity)
        for ranked, path in ((2, 3), (1, 2), (0, 1)):
            ctx.solve_set_ranked(ranked)
            for policy in (A.POLICY_NONE, A.POLICY_PRIORITY_EXHAUSTIVE, A.POLICY_PRIORITY_ROUND_ROBIN, A.POLICY_ROUND_ROBIN):
                for dbe in (False, True):
                    ctx.analyze_grid_device(R, B)
                    acc, chosen = ctx.solve_grid(unlimited=False, delayed_best_effort=dbe, policy=policy)
                    assert ctx.solve_greedy_path() == path
                    o_recs, o_feas = ref.copy_records(wva, recs, feas)
                    w_acc, w_chosen = oracle.solve(img, o_recs, o_feas, unlimited=False, delayed_best_effort=dbe, policy=policy)
                    assert np.array_equal(acc, w_acc), (ranked, policy, dbe)
                    _records_equal(chosen, w_chosen)
                    cnt, cst = ctx.allocate_by_type()
                    w_cnt, w_cst = oracle.allocate_by_type(img, w_acc, w_chosen)
                    assert np.array_equal(cnt, w_cnt) and cst.tobytes() == w_cst.tobytes()
                    assert (cnt <= img.type_capacity).all()
                    # consumed: a second limited solve needs a new sweep
                    with pytest.raises(WvaError) as e:
                        ctx.solve_grid(unlimited=False, policy=policy)
                    assert e.value.code == A.ESTATE
    finally:
        _reset(ctx, img)


def test_state_errors(wva, oracle, ctx):
    from inferno_autoscaler_b200.binding import WvaError
    img = wva.synth.make_system(24, 3, seed=7, n_types=2)
    o_pairs, o_feas, _ = oracle.analyze_pairs(img)
    w_acc, w_chosen = oracle.solve(img, o_pairs, o_feas, unlimited=True)

    def estate(f, *args, **kw):
        with pytest.raises(WvaError) as e:
            f(*args, **kw)
        assert e.value.code == wva.abi.ESTATE

    def pair_solve_ok():
        ctx.analyze_pairs(download=False)
        acc, chosen = ctx.solve(unlimited=True)
        assert np.array_equal(acc, w_acc) and chosen.equal_bits(w_chosen)[0]

    try:
        ctx.upload(img)
        ctx.grid_set_pair_winners(True)
        estate(ctx.solve_grid)                                    # before any sweep
        estate(ctx.grid_pairs_fetch)
        pair_solve_ok()
        ctx.grid_set_pair_winners(False)
        ctx.analyze_grid(8, 32)
        estate(ctx.solve_grid)                                    # after a sweep with the option off
        pair_solve_ok()
        ctx.grid_set_pair_winners(True)
        ctx.analyze_grid(8, 32)
        ctx.solve_grid(unlimited=True)
        ctx.update_servers(0, img.take(range(2)))                 # an image update
        estate(ctx.solve_grid)
        pair_solve_ok()
        ctx.analyze_grid(8, 32)
        ctx.analyze_pairs(download=False)
        ctx.solve_grid(unlimited=False, policy=wva.abi.POLICY_PRIORITY_EXHAUSTIVE)
        estate(ctx.solve_grid)                                    # consumed by a limited solve
        estate(ctx.grid_pairs_fetch)
        acc, chosen = ctx.solve(unlimited=True)                   # the pair records are untouched
        assert np.array_equal(acc, w_acc) and chosen.equal_bits(w_chosen)[0]
    finally:
        _reset(ctx, img)


# ---- two GPUs -------------------------------------------------------------------------------------------------

def _image(wva):
    return wva.synth.make_system(61, 4, seed=93, n_types=2, max_pair_batch=128)


def _one_rank_reference(wva, oracle, img, R, B, policy):
    """the whole system on one device: sweep records, limited solve, totals"""
    from inferno_autoscaler_b200 import binding
    ctx = binding.Context(0)
    try:
        ctx.upload(img)
        ctx.grid_set_pair_winners(True)
        ctx.analyze_grid(R, B)
        recs, feas = ctx.grid_pairs_fetch()
        acc, chosen = ctx.solve_grid(unlimited=False, policy=policy)
        cnt, cst = ctx.allocate_by_type()
    finally:
        ctx.close()
    o_recs, o_feas = ref.copy_records(wva, recs, feas)
    w_acc, w_chosen = oracle.solve(img, o_recs, o_feas, unlimited=False, policy=policy)
    assert np.array_equal(acc, w_acc) and chosen.equal_bits(w_chosen)[0]
    return recs, feas, acc, chosen, cnt, cst


def _caps(wva, img, R, B):
    from inferno_autoscaler_b200 import binding
    ctx = binding.Context(0)
    try:
        ctx.upload(img)
        ctx.grid_set_pair_winners(True)
        ctx.analyze_grid(R, B)
        acc, chosen = ctx.solve_grid(unlimited=True)
    finally:
        ctx.close()
    wva.synth.set_capacity_from_demand(img, acc, chosen.num_replicas, fraction=0.6)


def _worker(rank, world, port, q):
    sys.path.insert(0, ROOT)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    os.environ["MASTER_ADDR"] = "127.0.0.1"; os.environ["MASTER_PORT"] = str(port)
    import torch.distributed as dist
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    ok = False
    try:
        import wva_import
        wva = wva_import.load()
        from inferno_autoscaler_b200 import binding, distributed as D
        import oracle
        R, B = 8, 32
        policy = wva.abi.POLICY_PRIORITY_ROUND_ROBIN
        img = _image(wva)
        box = [None]
        if rank == 0:                     # caps and the one-device result come from rank 0's device
            _caps(wva, img, R, B)
            _, _, w_acc, w_chosen, w_cnt, w_cst = _one_rank_reference(wva, oracle, img, R, B, policy)
            box = [(img.type_capacity.copy(), w_acc, w_chosen.as_dict(), w_cnt, w_cst)]
        dist.broadcast_object_list(box, src=0)
        img.type_capacity[:] = box[0][0]
        box = [box[0][1:]]
        w_acc, w_ch, w_cnt, w_cst = box[0]
        ctx = binding.Context(rank)
        D.attach_library_comm(ctx, torch.device("cuda", rank))
        ctx.upload(img); ctx.comm_shard()
        ctx.grid_set_pair_winners(True)
        ctx.analyze_grid(R, B)
        acc, chosen = ctx.solve_grid(unlimited=False, policy=policy)       # gathers the sweep records itself
        ok = np.array_equal(acc, w_acc) and all(np.array_equal(getattr(chosen, k).view(np.uint8), v.view(np.uint8))
                                                 for k, v in w_ch.items())
        cnt, cst = ctx.allocate_by_type()                                  # global totals
        ok = ok and np.array_equal(cnt, w_cnt) and np.allclose(cst, w_cst, rtol=1e-5)
        ctx.comm_destroy()
        ctx.close()
    finally:
        q.put((rank, bool(ok)))
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus_comm_solve_grid():
    c = mp.get_context("spawn")
    q = c.Queue()
    port = 29800 + (os.getpid() % 1000)
    procs = [c.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]


def _group_case(wva, oracle, n_dev):
    from inferno_autoscaler_b200 import binding
    R, B = 8, 32
    img = _image(wva)
    _caps(wva, img, R, B)
    for policy in (wva.abi.POLICY_NONE, wva.abi.POLICY_PRIORITY_EXHAUSTIVE):
        w_recs, w_feas, w_acc, w_chosen, w_cnt, w_cst = _one_rank_reference(wva, oracle, img, R, B, policy)
        g = binding.Group(list(range(n_dev)))
        try:
            g.upload(img)
            g.grid_set_pair_winners(True)
            g.analyze(R, B)
            recs, feas = g.grid_pairs_fetch()
            assert np.array_equal(feas, w_feas) and recs.equal_bits(w_recs)[0]
            acc, chosen = g.solve_grid(unlimited=False, policy=policy)
            assert np.array_equal(acc, w_acc) and chosen.equal_bits(w_chosen)[0]
            cnt, cst = g.allocate_by_type()
            assert np.array_equal(cnt, w_cnt) and np.allclose(cst, w_cst, rtol=1e-5)
        finally:
            g.close()


def test_group_one_device_solve_grid(wva, oracle):
    _group_case(wva, oracle, 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_group_two_devices_solve_grid(wva, oracle):
    _group_case(wva, oracle, 2)
