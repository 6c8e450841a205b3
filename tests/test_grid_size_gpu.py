"""GPU: wva_grid_pairs_size -- QueueAnalyzer.Size for every per-pair sweep record at its own batch size, against the
oracle's queue_size (tests/grid_size_ref.sized_records).

  1. config 2, every record, certified-tails modes 1 and 0: status bytes, sized rates bit for bit, other fields unchanged;
  2. both paths: the thread path (wva_pairs_set_warp_max 0) gives the same bytes; records above the warp's shared-memory
     slice (b_max > 3072) go to the fallback and still equal the oracle;
  3. config 3 (all 8 000 pairs) and a 2 000-server slice of config 4;
  4. overflow-rescale chains: the oracle's rescale counter grows while it sizes the records;
  5. solves over sized and unsized records choose the same; the chosen records carry the sized rate;
  6. lifetime: WVA_ESTATE cases, sizing twice, the pair-record path unaffected;
  7. two GPUs / wva_group."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

import grid_size_ref as ref

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32
OTHER_FIELDS = ("acc", "num_replicas", "batch_size", "cost", "value", "itl", "ttft", "rho")


@pytest.fixture
def sctx(ctx):
    """the session context, back to its defaults afterwards"""
    yield ctx
    ctx.grid_set_pair_winners(False)
    ctx.set_certified_tails(1)
    ctx.pairs_set_warp_max(1 << 22)
    ctx.solve_set_ranked(2)


@pytest.fixture(scope="module")
def threads(oracle):
    return max(1, oracle.hardware_threads())


def _bits(x):
    return x.view(np.uint32) if x.dtype == np.float32 else x


def _sweep_and_size(ctx, R, B):
    """sweep with pair winners on, then size: (records before, feasible, records after, status)"""
    ctx.grid_set_pair_winners(True)
    ctx.analyze_grid_device(R, B)
    before, fe = ctx.grid_pairs_fetch()
    status = ctx.grid_pairs_size()
    after, fe2 = ctx.grid_pairs_fetch()
    assert np.array_equal(fe, fe2)
    return before, fe, after, status


def _check_against_oracle(wva, oracle, img, before, fe, after, status, threads):
    want, w_status = ref.sized_records(wva, oracle, img, before, fe, threads=threads)
    assert np.array_equal(status, w_status)
    assert np.array_equal(_bits(after.max_arrv_rate_per_replica), _bits(want.max_arrv_rate_per_replica))
    for name in OTHER_FIELDS:
        assert np.array_equal(_bits(getattr(after, name)), _bits(getattr(before, name))), name
    return w_status


def test_config2_every_record_equals_oracle(wva, oracle, sctx, threads):
    img, c = wva.synth.baseline_config(2)
    sctx.upload(img)
    for mode in (1, 0):
        sctx.set_certified_tails(mode)
        before, fe, after, status = _sweep_and_size(sctx, c["r_max"], c["b_max"])
        w_status = _check_against_oracle(wva, oracle, img, before, fe, after, status, threads)
        assert (w_status == 1).sum() > 0 and np.array_equal(w_status > 0, fe > 0)
        sized = w_status == 1
        assert (after.max_arrv_rate_per_replica[sized] != before.max_arrv_rate_per_replica[sized]).any()


def test_thread_path_same_bytes(wva, sctx):
    img, c = wva.synth.baseline_config(2)
    sctx.upload(img)
    _, _, warp, w_status = _sweep_and_size(sctx, c["r_max"], c["b_max"])
    sctx.pairs_set_warp_max(0)
    _, _, thr, t_status = _sweep_and_size(sctx, c["r_max"], c["b_max"])
    assert np.array_equal(w_status, t_status)
    ok, field = thr.equal_bits(warp)
    assert ok, field


def _large_batch_image(wva):
    """tiny beta / delta (the parameters of test_pairs_overflow_rescale_path): a batch of n serves about n times one
    request's rate, so with one replica the cheapest feasible batch grows with the load, past 3072 for the larger loads,
    and the chains take the overflow-rescale branches"""
    img = wva.synth.make_system(8, 1, seed=5, max_pair_batch=0)
    img.perf_alpha[:] = 20.0; img.perf_beta[:] = 1e-4; img.perf_gamma[:] = 10.0; img.perf_delta[:] = 1e-7
    img.perf_valid[:] = 1; img.srv_target_valid[:] = 1
    img.srv_arrival_rpm[:] = [2e5, 6e5, 1.0e6, 1.15e6, 1.3e6, 1.45e6, 1.6e6, 2.0e6]
    img.srv_in_tokens[:] = 64; img.srv_out_tokens[:] = 8
    img.srv_slo_itl[:] = 200.0; img.srv_slo_ttft[:] = 2000.0; img.srv_slo_tps[:] = 0.0
    img.srv_keep_acc[:] = 0; img.srv_min_replicas[:] = 0; img.srv_max_batch[:] = 0
    return img


@pytest.mark.parametrize("warp_max", [1 << 22, 0])
def test_large_batches_fallback_and_overflow_rescale(wva, oracle, sctx, threads, warp_max):
    img = _large_batch_image(wva)
    sctx.upload(img)
    sctx.pairs_set_warp_max(warp_max)
    before, fe, after, status = _sweep_and_size(sctx, 1, 4096)
    assert (before.batch_size[fe > 0] > 3072).any(), "no record larger than the warp's shared-memory slice"
    ev0 = oracle.rescale_events()
    w_status = _check_against_oracle(wva, oracle, img, before, fe, after, status, threads)
    assert oracle.rescale_events() > ev0, "the records' Size never took an overflow-rescale branch"
    assert (w_status == 1).any()


@pytest.mark.parametrize("which", ["config3", "config4_slice"])
def test_measured_sizes_equal_oracle(wva, oracle, sctx, threads, which):
    if which == "config3":
        img, c = wva.synth.baseline_config(3)
        first, count = 0, img.S
    else:
        c = wva.synth.CONFIGS[4]
        img = wva.synth.make_system(c["S"], c["A"], seed=4, n_types=c["T"])
        first, count = 4000, 2000
    sctx.upload(img)
    sctx.set_shard(first, count)
    before, fe, after, status = _sweep_and_size(sctx, c["r_max"], c["b_max"])
    lo, hi = first * img.A, (first + count) * img.A
    assert (status[:lo] == 0).all() and (status[hi:] == 0).all()
    _check_against_oracle(wva, oracle, img, before, fe, after, status, threads)
    assert int((status == 1).sum()) > 1000
    print(which, "records:", int(fe.sum()), "status histogram:", np.bincount(status, minlength=3).tolist())


def test_solves_unchanged_and_carry_sized_rate(wva, sctx):
    img, c = wva.synth.baseline_config(3)
    R, B = c["r_max"], c["b_max"]
    A = wva.abi
    sctx.upload(img)
    sctx.grid_set_pair_winners(True)
    sctx.analyze_grid_device(R, B)
    u_acc, u_chosen = sctx.solve_grid(unlimited=True)
    sctx.grid_pairs_size()
    sized, _ = sctx.grid_pairs_fetch()
    s_acc, s_chosen = sctx.solve_grid(unlimited=True)

    def same(acc1, ch1, acc2, ch2):
        assert np.array_equal(acc1, acc2)
        for name in ("num_replicas", "batch_size", "cost", "value"):
            assert np.array_equal(_bits(getattr(ch1, name)), _bits(getattr(ch2, name))), name

    def carries(acc, ch):
        has = acc >= 0
        gi = np.flatnonzero(has) * img.A + acc[has]
        assert np.array_equal(_bits(ch.max_arrv_rate_per_replica[has]), _bits(sized.max_arrv_rate_per_replica[gi]))

    same(u_acc, u_chosen, s_acc, s_chosen)
    carries(s_acc, s_chosen)
    wva.synth.set_capacity_from_demand(img, u_acc, u_chosen.num_replicas, fraction=0.6)
    sctx.set_capacity(img.type_capacity)
    for ranked, path in ((2, 3), (1, 2), (0, 1)):
        sctx.solve_set_ranked(ranked)
        for policy in (A.POLICY_NONE, A.POLICY_PRIORITY_EXHAUSTIVE, A.POLICY_PRIORITY_ROUND_ROBIN, A.POLICY_ROUND_ROBIN):
            sctx.analyze_grid_device(R, B)
            acc1, ch1 = sctx.solve_grid(unlimited=False, policy=policy)
            sctx.analyze_grid_device(R, B)
            sctx.grid_pairs_size()
            acc2, ch2 = sctx.solve_grid(unlimited=False, policy=policy)
            assert sctx.solve_greedy_path() == path
            same(acc1, ch1, acc2, ch2)
            carries(acc2, ch2)


def test_lifetime(wva, oracle, sctx):
    from inferno_autoscaler_b200.binding import WvaError
    img = wva.synth.make_system(24, 3, seed=7, n_types=2)
    o_pairs, o_feas, _ = oracle.analyze_pairs(img)
    w_acc, w_chosen = oracle.solve(img, o_pairs, o_feas, unlimited=True)

    def estate():
        with pytest.raises(WvaError) as e:
            sctx.grid_pairs_size()
        assert e.value.code == wva.abi.ESTATE

    def pair_solve_ok():
        sctx.analyze_pairs(download=False)
        acc, chosen = sctx.solve(unlimited=True)
        assert np.array_equal(acc, w_acc) and chosen.equal_bits(w_chosen)[0]

    sctx.upload(img)
    sctx.grid_set_pair_winners(True)
    estate()                                                  # before any sweep
    sctx.grid_set_pair_winners(False)
    sctx.analyze_grid(8, 32)
    estate()                                                  # option off
    sctx.grid_set_pair_winners(True)
    sctx.analyze_grid(8, 32)
    st1 = sctx.grid_pairs_size()
    r1, f1 = sctx.grid_pairs_fetch()
    st2 = sctx.grid_pairs_size()                              # sizing twice: same bytes
    r2, f2 = sctx.grid_pairs_fetch()
    assert np.array_equal(st1, st2) and np.array_equal(f1, f2) and r1.equal_bits(r2)[0]
    pair_solve_ok()
    sctx.update_servers(0, img.take(range(2)))                # image update
    estate()
    sctx.analyze_grid(8, 32)
    sctx.set_shard(0, 12)                                     # shard change
    estate()
    sctx.set_shard(0, img.S)
    sctx.analyze_grid(8, 32)
    sctx.grid_pairs_size()
    sctx.solve_grid(unlimited=False, policy=wva.abi.POLICY_PRIORITY_EXHAUSTIVE)
    estate()                                                  # consumed by a limited solve
    pair_solve_ok()


def test_group_one_device_equals_context(wva, sctx):
    _group_case(wva, sctx, 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_group_two_devices_equals_context(wva, sctx):
    _group_case(wva, sctx, 2)


def _image(wva):
    return wva.synth.make_system(61, 4, seed=93, n_types=2, max_pair_batch=128)


def _group_case(wva, ctx, n_dev):
    from inferno_autoscaler_b200 import binding
    R, B = 8, 32
    img = _image(wva)
    ctx.upload(img)
    ctx.grid_set_pair_winners(True)
    ctx.analyze_grid(R, B)
    w_status = ctx.grid_pairs_size()
    w_recs, w_fe = ctx.grid_pairs_fetch()
    g = binding.Group(list(range(n_dev)))
    try:
        g.upload(img)
        g.grid_set_pair_winners(True)
        g.analyze(R, B)
        status = g.grid_pairs_size()
        recs, fe = g.grid_pairs_fetch()
        assert np.array_equal(status, w_status) and np.array_equal(fe, w_fe) and recs.equal_bits(w_recs)[0]
    finally:
        g.close()


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
        R, B = 8, 32
        policy = wva.abi.POLICY_PRIORITY_ROUND_ROBIN
        img = _image(wva)
        box = [None]
        if rank == 0:                     # caps and the one-device result come from rank 0's device
            c = binding.Context(0)
            try:
                c.upload(img)
                c.grid_set_pair_winners(True)
                c.analyze_grid(R, B)
                acc, chosen = c.solve_grid(unlimited=True)
                wva.synth.set_capacity_from_demand(img, acc, chosen.num_replicas, fraction=0.6)
                c.set_capacity(img.type_capacity)
                c.analyze_grid(R, B)
                c.grid_pairs_size()
                w_acc, w_chosen = c.solve_grid(unlimited=False, policy=policy)
            finally:
                c.close()
            box = [(img.type_capacity.copy(), w_acc, w_chosen.as_dict())]
        dist.broadcast_object_list(box, src=0)
        img.type_capacity[:] = box[0][0]
        w_acc, w_ch = box[0][1], box[0][2]
        ctx = binding.Context(rank)
        D.attach_library_comm(ctx, torch.device("cuda", rank))
        ctx.upload(img); ctx.comm_shard()
        ctx.grid_set_pair_winners(True)
        ctx.analyze_grid(R, B)
        ctx.grid_pairs_size()                                          # this rank's rows
        acc, chosen = ctx.solve_grid(unlimited=False, policy=policy)   # the gather moves the sized rates
        ok = np.array_equal(acc, w_acc) and all(np.array_equal(getattr(chosen, k).view(np.uint8), v.view(np.uint8))
                                                 for k, v in w_ch.items())
        ctx.comm_destroy()
        ctx.close()
    finally:
        q.put((rank, bool(ok)))
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus_comm_solve_over_sized_records():
    c = mp.get_context("spawn")
    q = c.Queue()
    port = 29900 + (os.getpid() % 1000)
    procs = [c.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]
