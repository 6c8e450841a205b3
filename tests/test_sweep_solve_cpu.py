"""CPU-only: the sweep's per-(server, accelerator) winners as solver input, on the oracle side.

The per-pair records (tests/sweep_pair_ref.py) are reduced from the oracle's per-candidate sweep; a server's
sweep winner must be the best of its pairs' records, and the unlimited solve over those records must pick it."""
import numpy as np
import pytest

import sweep_pair_ref as ref

F = np.float32
MAX_F32 = np.finfo(np.float32).max


def _sweep(wva, oracle, seed):
    img = wva.synth.make_system(12, 3, seed=seed, n_types=2, max_pair_batch=64)
    R, B = 8, 64
    best, cube, status, _ = oracle.analyze_grid(img, R, B, want_cube=True, threads=max(1, oracle.hardware_threads()))
    recs, feas = ref.pair_records(wva, oracle, img, R, B, cube, status)
    return img, best, recs, feas


@pytest.mark.parametrize("seed", [3, 17, 29])
def test_server_best_is_min_of_pair_bests(wva, oracle, seed):
    img, best, recs, feas = _sweep(wva, oracle, seed)
    acc, rep, bat, gi = ref.best_of_pairs(recs, feas, img.S, img.A)
    assert np.array_equal(acc, best["acc"])
    has = acc >= 0
    assert has.sum() >= 3 and feas.sum() > has.sum()           # the records carry alternatives, not just winners
    assert np.array_equal(rep[has], best["replicas"][has]) and np.array_equal(bat[has], best["batch"][has])
    for f in ("cost", "value", "itl", "ttft", "rho"):
        assert np.array_equal(getattr(recs, f)[gi[has]].view(np.uint32), best[f][has].view(np.uint32)), f
    # infeasible pairs hold the empty record
    off = feas == 0
    assert (recs.acc[off] == ref.ACC_NONE).all() and (recs.num_replicas[off] == 0).all() and (recs.cost[off] == 0).all()


@pytest.mark.parametrize("seed", [3, 17, 29])
def test_unlimited_solve_on_sweep_records_picks_the_sweep_winner(wva, oracle, seed):
    img, best, recs, feas = _sweep(wva, oracle, seed)
    chosen_acc, chosen = oracle.solve(img, recs, feas, unlimited=True)
    win = (best["acc"] >= 0) & (best["value"] < MAX_F32)
    assert win.sum() >= 3
    assert np.array_equal(chosen_acc[win], best["acc"][win])
    assert np.array_equal(chosen.num_replicas[win], best["replicas"][win].astype(np.int64))
    assert np.array_equal(chosen.batch_size[win], best["batch"][win].astype(np.int64))
    assert (chosen_acc[~win] == -1).all()


def test_exports_list_the_sweep_solve_calls(wva):
    from inferno_autoscaler_b200 import binding
    for name in ("wva_grid_set_pair_winners", "wva_grid_pairs_fetch", "wva_grid_pairs_fetch_arrays", "wva_solve_grid",
                 "wva_solve_grid_arrays", "wva_group_grid_pairs_fetch", "wva_group_solve_grid"):
        assert name in binding.EXPORTS
