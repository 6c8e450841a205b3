"""Per-(server, accelerator) sweep winners restated from the oracle's per-candidate results.

Test helper (not collected): the oracle evaluates every sweep candidate through the reference API
(oracle.analyze_grid / grid_candidates) and gives every sweep row's transition-penalty value
(oracle.grid_row_values); this module reduces those per pair and writes the wva_alloc_soa records that
wva_grid_pairs_fetch returns, field for field (include/wva_b200.h, wva_grid_set_pair_winners):

  record of pair (s, a) = the feasible candidate with a non-NaN value and the smallest (value, r, b)
  acc = a, num_replicas = r, batch_size = b, cost = acc.Cost * float32(numInstances * r),
  value, itl, ttft = wait + prefill, rho as in wva_grid_best,
  max_arrv_rate_per_replica = (totalRate / float32(r)) / 1000 (the rate the candidate was analysed at);
  no such candidate: feasible = 0 and the empty record (acc = -1, zeros).
"""
import numpy as np

F = np.float32
ACC_NONE = -1


def total_rate(img, s):
    """allocation.go:134-139 in float32: arrival rpm / 60, or slo_tps / out_tokens when the TPS target is set"""
    tps = img.srv_slo_tps[s].astype(F)
    rpm = img.srv_arrival_rpm[s].astype(F)
    out = img.srv_out_tokens[s].astype(F)
    with np.errstate(divide="ignore", invalid="ignore"):
        return np.where(tps == F(0), rpm / F(60), tps / out).astype(F)


def candidate_fields(img, s, a, r, b, value, metrics):
    """record fields of the candidates (s, a, r, b) (global server index) from their metrics and row values"""
    s, a, r, b = (np.asarray(x, dtype=np.int64) for x in (s, a, r, b))
    cnt = img.perf_acc_count[img.srv_model[s].astype(np.int64) * img.A + a].astype(np.int64)
    ninst = np.where(cnt <= 0, 1, cnt)
    rate = total_rate(img, s)
    return dict(acc=a.astype(np.int32), num_replicas=r, batch_size=b,
                cost=(img.acc_cost[a].astype(F) * (ninst * r).astype(F)).astype(F),
                value=np.asarray(value, dtype=F),
                itl=metrics["avg_token_time"].astype(F),
                ttft=(metrics["avg_wait_time"] + metrics["avg_prefill_time"]).astype(F),
                rho=metrics["rho"].astype(F),
                max_arrv_rate_per_replica=((rate / r.astype(F)).astype(F) / F(1000)).astype(F))


def empty_records(wva, img, s0=0, s1=None):
    """AllocArrays[S*A] + feasible[S*A] as a fetch leaves them before any pair is found: shard rows empty
    (acc = -1), rows of other shards zero"""
    s1 = img.S if s1 is None else s1
    recs = wva.abi.AllocArrays(img.S * img.A)
    recs.acc[s0 * img.A:s1 * img.A] = ACC_NONE
    return recs, np.zeros(img.S * img.A, dtype=np.uint8)


def copy_records(wva, recs, feasible):
    """a copy for oracle.solve, whose best-effort scaling writes the records in place"""
    out = wva.abi.AllocArrays(recs.n)
    for name, _ in wva.abi.ALLOC_FIELDS:
        getattr(out, name)[:] = getattr(recs, name)
    return out, feasible.copy()


def fill(recs, feasible, gi, fields):
    for name, v in fields.items():
        getattr(recs, name)[gi] = v
    feasible[gi] = 1


def pair_records(wva, oracle, img, R, B, cube, status, s0=0, s1=None):
    """the records of servers [s0, s1) from the oracle's full cube / status of that slice"""
    s1 = img.S if s1 is None else s1
    ns, A = s1 - s0, img.A
    vals = oracle.grid_row_values(img, R, s0, s1)                       # [ns, A, R]
    feas = ((status.reshape(ns, A, R, B) & wva.abi.CAND_FEASIBLE) != 0) & ~np.isnan(vals)[..., None]
    row_has = feas.any(-1)
    first_b = feas.argmax(-1)                                           # within a row the key grows with b
    v = np.where(row_has, vals, np.inf)
    r_ix = v.argmin(-1)                                                 # smallest value, then smallest r
    has = row_has.any(-1)
    sl, a = np.nonzero(has)
    r = r_ix[sl, a]
    assert row_has[sl, a, r].all()
    b = first_b[sl, a, r]
    ci = ((sl.astype(np.int64) * A + a) * R + r) * B + b
    recs, feasible = empty_records(wva, img, s0, s1)
    fill(recs, feasible, (sl + s0) * A + a, candidate_fields(img, sl + s0, a, r + 1, b + 1, vals[sl, a, r], cube[ci]))
    return recs, feasible


def best_of_pairs(recs, feasible, S, A):
    """per-server minimum of the pair records by (value, a, r, b): (acc, r, b, index into recs) with acc = -1 where none"""
    acc = np.full(S, -1, dtype=np.int32)
    rep = np.zeros(S, dtype=np.int64)
    bat = np.zeros(S, dtype=np.int64)
    gi = np.full(S, -1, dtype=np.int64)
    for s in range(S):
        best = None
        for a in range(A):
            i = s * A + a
            if not feasible[i]:
                continue
            k = (float(recs.value[i]), a, int(recs.num_replicas[i]), int(recs.batch_size[i]))
            if best is None or k < best[0]:
                best = (k, i)
        if best is not None:
            acc[s], rep[s], bat[s], gi[s] = best[0][1], best[0][2], best[0][3], best[1]
    return acc, rep, bat, gi
