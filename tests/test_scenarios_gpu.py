"""GPU: wva_analyze_scenarios -- Server.Calculate -> unlimited Solve -> AllocateByType under many load scenarios, one
Size per pair, against the oracle run once per scenario on a copy of the image whose srv_arrival_rpm is that row.

  1. config 2, ~40 scenarios (multipliers 0 .. 8 of the image's rates, its own rates, all zeros, negative entries),
     certified-tails modes 1 and 0: every record and feasible byte, every decision, count and cost bit for bit;
  2. the scenario equal to the image's own rates gives what wva_analyze_pairs + wva_solve + wva_allocate_by_type give;
  3. warp path against thread path (wva_pairs_set_warp_max 0); pairs above the warp's shared-memory slice
     (srv_max_batch > 3072) and overflow-rescale chains (the oracle's rescale counter grows), both against the oracle;
  4. config 3 (all 8 000 pairs, 16 scenarios) and a 2 000-server slice of config 4 (8 scenarios);
  5. a TPS-target server's positive scenarios all get the same record;
  6. state: WVA_ESTATE / WVA_EINVAL cases, the resident results untouched, launches independent of the scenario count;
  7. wva_group and two GPUs against one rank."""
import ctypes as C
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
F = np.float32


@pytest.fixture
def sctx(ctx):
    """the session context, back to its defaults afterwards"""
    yield ctx
    ctx.grid_set_pair_winners(False)
    ctx.set_certified_tails(1)
    ctx.pairs_set_warp_max(1 << 22)


@pytest.fixture(scope="module")
def threads(oracle):
    return max(1, oracle.hardware_threads())


def _rows(allocs, lo, hi):
    """records [lo, hi) of an AllocArrays as a new AllocArrays"""
    from inferno_autoscaler_b200 import abi
    out = abi.AllocArrays(hi - lo)
    for name, _ in abi.ALLOC_FIELDS:
        getattr(out, name)[:] = getattr(allocs, name)[lo:hi]
    return out


def _scaled(img, mults):
    return (img.srv_arrival_rpm.astype(np.float64)[None, :] * np.asarray(mults, dtype=np.float64)[:, None]).astype(F)


def _config2_rates(img, seed=11):
    mults = np.concatenate([[0.0], np.arange(1, 9) / 8.0, np.arange(1.25, 8.01, 0.25)])
    rates = _scaled(img, mults)
    neg = img.srv_arrival_rpm.copy()
    rng = np.random.default_rng(seed)
    neg[rng.uniform(0, 1, img.S) < 0.4] *= -1.0
    neg[0] = -1.0
    return np.vstack([rates, img.srv_arrival_rpm[None, :], np.zeros((1, img.S), F), neg[None, :]]).astype(F)


def _oracle_scenario(oracle, img, row, threads, first=0, count=None):
    """(pairs, feasible, chosen_acc, chosen, count, cost) of servers [first, first+count) with arrival rates `row`"""
    count = img.S if count is None else count
    sub = img.shard(first, count)
    sub.srv_arrival_rpm[:] = row[first:first + count]
    pairs, fe, _ = oracle.analyze_pairs(sub, threads=threads)
    acc, chosen = oracle.solve(sub, pairs, fe, unlimited=True)
    cnt, cst = oracle.allocate_by_type(sub, acc, chosen)
    return pairs, fe, acc, chosen, cnt, cst


def _check_against_oracle(wva, oracle, ctx, img, rates, out, threads, first=0, count=None):
    count = img.S if count is None else count
    acc, chosen, cnt, cst = out
    A = img.A
    lo, hi = first * A, (first + count) * A
    for l in range(rates.shape[0]):
        o_pairs, o_fe, o_acc, o_chosen, o_cnt, o_cst = _oracle_scenario(oracle, img, rates[l], threads, first, count)
        recs, fe = ctx.scenario_pairs_fetch(l)
        assert np.array_equal(fe[lo:hi], o_fe), "scenario %d: feasible" % l
        ok, field = _rows(recs, lo, hi).equal_bits(o_pairs)
        assert ok, "scenario %d: pair field %s" % (l, field)
        assert np.array_equal(acc[l, first:first + count], o_acc), "scenario %d: decisions" % l
        ok, field = _rows(chosen, l * img.S + first, l * img.S + first + count).equal_bits(o_chosen)
        assert ok, "scenario %d: chosen field %s" % (l, field)
        assert np.array_equal(cnt[l], o_cnt) and cst[l].tobytes() == o_cst.tobytes(), "scenario %d: totals" % l


@pytest.mark.parametrize("mode", [1, 0])
def test_config2_every_scenario_equals_oracle(wva, oracle, sctx, threads, mode):
    img, _ = wva.synth.baseline_config(2)
    sctx.upload(img)
    sctx.set_certified_tails(mode)
    rates = _config2_rates(img)
    assert 38 <= rates.shape[0] <= 42
    out = sctx.analyze_scenarios(rates)
    _check_against_oracle(wva, oracle, sctx, img, rates, out, threads)
    assert (out[0] >= 0).any() and (out[2] > 0).any()
    assert sctx.phase_usec(wva.abi.PHASE_SCENARIOS) > 0


def test_own_rates_equal_resident_path(wva, sctx):
    img, _ = wva.synth.baseline_config(2)
    sctx.upload(img)
    pairs, fe = sctx.analyze_pairs()
    acc, chosen = sctx.solve(unlimited=True)
    cnt, cst = sctx.allocate_by_type()
    rates = _scaled(img, [0.5, 1.0, 2.0])
    s_acc, s_chosen, s_cnt, s_cst = sctx.analyze_scenarios(rates)
    recs, s_fe = sctx.scenario_pairs_fetch(1)
    assert np.array_equal(s_fe, fe) and recs.equal_bits(pairs)[0]
    assert np.array_equal(s_acc[1], acc) and _rows(s_chosen, img.S, 2 * img.S).equal_bits(chosen)[0]
    assert np.array_equal(s_cnt[1], cnt) and s_cst[1].tobytes() == cst.tobytes()


def _fetch_all(ctx, L):
    return [ctx.scenario_pairs_fetch(l) for l in range(L)]


def _same_results(a, b, ra, rb):
    assert np.array_equal(a[0], b[0]) and a[1].equal_bits(b[1])[0]
    assert np.array_equal(a[2], b[2]) and a[3].tobytes() == b[3].tobytes()
    for (r1, f1), (r2, f2) in zip(ra, rb):
        assert np.array_equal(f1, f2)
        ok, field = r1.equal_bits(r2)
        assert ok, field


def test_thread_path_same_bytes(wva, sctx):
    img, _ = wva.synth.baseline_config(2)
    sctx.upload(img)
    rates = _config2_rates(img)
    warp = sctx.analyze_scenarios(rates)
    w_recs = _fetch_all(sctx, rates.shape[0])
    sctx.pairs_set_warp_max(0)
    thr = sctx.analyze_scenarios(rates)
    t_recs = _fetch_all(sctx, rates.shape[0])
    _same_results(warp, thr, w_recs, t_recs)


def _large_batch_image(wva):
    """tiny beta / delta: a batch of n serves about n times one request's rate, so the ramp of a long chain grows past
    double range and takes the overflow-rescale branches; two servers carry a batch override above the warp's
    3 072-entry shared-memory slice"""
    img = wva.synth.make_system(8, 1, seed=5, max_pair_batch=0)
    img.perf_alpha[:] = 20.0; img.perf_beta[:] = 1e-4; img.perf_gamma[:] = 10.0; img.perf_delta[:] = 1e-7
    img.perf_valid[:] = 1; img.srv_target_valid[:] = 1
    img.srv_arrival_rpm[:] = [2e5, 6e5, 1.0e6, 1.15e6, 1.3e6, 1.45e6, 1.6e6, 2.0e6]
    img.srv_in_tokens[:] = 64; img.srv_out_tokens[:] = 8
    img.srv_slo_itl[:] = 200.0; img.srv_slo_ttft[:] = 2000.0; img.srv_slo_tps[:] = 0.0
    img.srv_keep_acc[:] = 0; img.srv_min_replicas[:] = 0
    img.srv_max_batch[:] = [4000, 3500, 1024, 2048, 0, 0, 0, 0]
    return img


@pytest.mark.parametrize("warp_max", [1 << 22, 0])
def test_large_batches_and_overflow_rescale(wva, oracle, sctx, threads, warp_max):
    img = _large_batch_image(wva)
    sctx.upload(img)
    sctx.pairs_set_warp_max(warp_max)
    rates = _scaled(img, [0.25, 0.5, 1.0, 2.0])
    out = sctx.analyze_scenarios(rates)
    recs = _fetch_all(sctx, rates.shape[0])
    assert any((r.batch_size[f > 0] > 3072).any() and (r.acc[f > 0] >= 0).any() for r, f in recs), \
        "no feasible record larger than the warp's shared-memory slice"
    ev0 = oracle.rescale_events()
    _check_against_oracle(wva, oracle, sctx, img, rates, out, threads)
    assert oracle.rescale_events() > ev0, "no scenario's CreateAllocation took an overflow-rescale branch"


def _tps_servers_share_records(img, recs, rates):
    tps = np.flatnonzero(img.srv_slo_tps > 0)
    assert len(tps) > 0
    A = img.A
    checked = 0
    for s in tps:
        pos = np.flatnonzero(rates[:, s] > 0)
        for l in pos[1:]:
            r0, f0 = recs[pos[0]]
            r1, f1 = recs[l]
            sl = slice(s * A, (s + 1) * A)
            assert np.array_equal(f0[sl], f1[sl])
            assert _rows(r0, s * A, (s + 1) * A).equal_bits(_rows(r1, s * A, (s + 1) * A))[0]
            checked += 1
    assert checked > 0


@pytest.mark.parametrize("which", ["config3", "config4_slice"])
def test_larger_configs_equal_oracle(wva, oracle, sctx, threads, which):
    if which == "config3":
        img, _ = wva.synth.baseline_config(3)
        first, count, L = 0, img.S, 16
    else:
        c = wva.synth.CONFIGS[4]
        img = wva.synth.make_system(c["S"], c["A"], seed=4, n_types=c["T"])
        first, count, L = 4000, 2000, 8
    sctx.upload(img)
    sctx.set_shard(first, count)
    mults = np.concatenate([[0.0, 1.0], np.geomspace(1.0 / 8.0, 8.0, L - 2)])
    rates = _scaled(img, mults)
    out = sctx.analyze_scenarios(rates)
    acc = out[0]
    assert (acc[:, :first] == -1).all() and (acc[:, first + count:] == -1).all()
    _check_against_oracle(wva, oracle, sctx, img, rates, out, threads, first, count)
    recs = _fetch_all(sctx, L)
    _tps_servers_share_records(img.shard(first, count), [(_rows(r, first * img.A, (first + count) * img.A),
                                                          f[first * img.A:(first + count) * img.A]) for r, f in recs],
                               rates[:, first:first + count])
    print(which, "feasible records per scenario:", [int(f.sum()) for _, f in recs])


def test_state_and_errors(wva, sctx):
    from inferno_autoscaler_b200 import binding
    A = wva.abi
    L_ = binding.lib()

    def code(fn):
        with pytest.raises(binding.WvaError) as e:
            fn()
        return e.value.code

    img = wva.synth.make_system(24, 3, seed=7, n_types=2)
    rates = _scaled(img, [0.5, 1.0, 3.0])
    fresh = binding.Context(0)
    try:
        fresh.image = img
        assert code(lambda: fresh.analyze_scenarios(rates)) == A.ESTATE          # no image uploaded
        assert code(lambda: fresh.scenario_pairs_fetch(0)) == A.ESTATE
    finally:
        fresh.close()

    sctx.upload(img)
    assert code(lambda: sctx.scenario_pairs_fetch(0)) == A.ESTATE                 # no call yet

    def raw(n, r):
        return L_.wva_analyze_scenarios(sctx._h, n, A.ptr(r, C.c_float), None, None, None, None)
    big = np.ones((1025, img.S), F)
    assert raw(0, rates) == A.EINVAL and raw(1025, big) == A.EINVAL
    for bad in (np.nan, np.inf, -np.inf):
        r = rates.copy()
        r[1, 5] = bad
        assert raw(3, r) == A.EINVAL

    # everything resident stays as it was
    sctx.grid_set_pair_winners(True)
    sctx.analyze(8, 32)
    p0, f0 = sctx.pairs_fetch()
    g0, gf0 = sctx.grid_pairs_fetch()
    acc0, ch0 = sctx.solve(unlimited=True)
    cnt0, cst0 = sctx.allocate_by_type()
    sctx.analyze_scenarios(rates)
    cnt1, cst1 = sctx.allocate_by_type()                                          # the solution is untouched
    assert np.array_equal(cnt0, cnt1) and cst0.tobytes() == cst1.tobytes()
    p1, f1 = sctx.pairs_fetch()
    g1, gf1 = sctx.grid_pairs_fetch()
    assert np.array_equal(f0, f1) and p0.equal_bits(p1)[0] and np.array_equal(gf0, gf1) and g0.equal_bits(g1)[0]
    ga, gch = sctx.solve_grid(unlimited=True)
    acc1, ch1 = sctx.solve(unlimited=True)
    assert np.array_equal(acc0, acc1) and ch0.equal_bits(ch1)[0]
    assert (ga >= 0).any()

    # the records stay until the next call, upload, update or shard change
    sctx.analyze_scenarios(rates)
    r_a, _ = sctx.scenario_pairs_fetch(2)
    sctx.analyze_pairs(download=False)
    r_b, _ = sctx.scenario_pairs_fetch(2)
    assert r_a.equal_bits(r_b)[0]
    with pytest.raises(binding.WvaError) as e:
        sctx.scenario_pairs_fetch(3)
    assert e.value.code == A.EINVAL
    sctx.update_servers(0, img.take(range(2)))
    assert code(lambda: sctx.scenario_pairs_fetch(0)) == A.ESTATE
    sctx.analyze_scenarios(rates)
    sctx.set_shard(0, 12)
    assert code(lambda: sctx.scenario_pairs_fetch(0)) == A.ESTATE
    sctx.analyze_scenarios(rates)
    sctx.upload(img)
    assert code(lambda: sctx.scenario_pairs_fetch(0)) == A.ESTATE


@pytest.mark.parametrize("warp_max", [1 << 22, 0])
def test_launches_independent_of_scenario_count(wva, sctx, warp_max):
    img, _ = wva.synth.baseline_config(2)
    sctx.upload(img)
    sctx.pairs_set_warp_max(warp_max)
    counts = []
    for L in (1, 32, 33, 300):
        rates = _scaled(img, np.linspace(0.5, 4.0, L))
        n0 = sctx.launch_count()
        sctx.analyze_scenarios(rates)
        counts.append(sctx.launch_count() - n0)
    assert len(set(counts)) == 1, counts


def _image(wva):
    return wva.synth.make_system(61, 4, seed=93, n_types=2, max_pair_batch=128)


def _rates61(img):
    rates = _scaled(img, [0.0, 0.25, 1.0, 2.5, 6.0])
    rates[4, ::7] = -5.0
    return rates


def test_group_one_device_equals_context(wva, sctx):
    _group_case(wva, sctx, 1)


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_group_two_devices_equals_context(wva, sctx):
    _group_case(wva, sctx, 2)


def _close_costs(a, b):
    return np.allclose(a, b, rtol=1e-5, atol=0.0)


def _group_case(wva, ctx, n_dev):
    from inferno_autoscaler_b200 import binding
    img = _image(wva)
    rates = _rates61(img)
    ctx.upload(img)
    w = ctx.analyze_scenarios(rates)
    w_recs = _fetch_all(ctx, rates.shape[0])
    g = binding.Group(list(range(n_dev)))
    try:
        g.upload(img)
        out = g.analyze_scenarios(rates)
        recs = [g.scenario_pairs_fetch(l) for l in range(rates.shape[0])]
        assert np.array_equal(out[0], w[0]) and out[1].equal_bits(w[1])[0] and np.array_equal(out[2], w[2])
        assert _close_costs(out[3], w[3]) if n_dev > 1 else out[3].tobytes() == w[3].tobytes()
        for (r1, f1), (r2, f2) in zip(recs, w_recs):
            assert np.array_equal(f1, f2) and r1.equal_bits(r2)[0]
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
        img = _image(wva)
        rates = _rates61(img)
        box = [None]
        if rank == 0:                     # the one-rank result comes from rank 0's device
            c = binding.Context(0)
            try:
                c.upload(img)
                acc, chosen, cnt, cst = c.analyze_scenarios(rates)
                recs = [c.scenario_pairs_fetch(l) for l in range(rates.shape[0])]
            finally:
                c.close()
            box = [(acc, chosen.as_dict(), cnt, cst, [(r.as_dict(), f) for r, f in recs])]
        dist.broadcast_object_list(box, src=0)
        w_acc, w_ch, w_cnt, w_cst, w_recs = box[0]
        ctx = binding.Context(rank)
        D.attach_library_comm(ctx, torch.device("cuda", rank))
        ctx.upload(img); ctx.comm_shard()
        acc, chosen, cnt, cst = ctx.analyze_scenarios(rates)
        S, A = img.S, img.A
        lo, hi = ctx.first, ctx.first + ctx.count
        ok = np.array_equal(acc[:, lo:hi], w_acc[:, lo:hi]) and np.array_equal(cnt, w_cnt) and _close_costs(cst, w_cst)
        for l in range(rates.shape[0]):
            sl = slice(l * S + lo, l * S + hi)
            ok = ok and all(np.array_equal(getattr(chosen, k)[sl].view(np.uint8), v[sl].view(np.uint8)) for k, v in w_ch.items())
            r, f = ctx.scenario_pairs_fetch(l)
            wr, wf = w_recs[l]
            ps = slice(lo * A, hi * A)
            ok = ok and np.array_equal(f[ps], wf[ps]) and all(np.array_equal(getattr(r, k)[ps].view(np.uint8), v[ps].view(np.uint8))
                                                             for k, v in wr.items())
        ctx.comm_destroy()
        ctx.close()
    finally:
        q.put((rank, bool(ok)))
        dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_gpus_comm_equals_one_rank():
    c = mp.get_context("spawn")
    q = c.Queue()
    port = 29950 + (os.getpid() % 1000)
    procs = [c.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = [q.get(timeout=600) for _ in procs]
    for p in procs:
        p.join(timeout=60)
    assert sorted(res) == [(0, True), (1, True)]
