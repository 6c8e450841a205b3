"""Expected results of wva_grid_pairs_size, restated from the oracle's QueueAnalyzer.Size.

Test helper (not collected): for each per-pair sweep record (s, a) of batch size b, the oracle's queue_size runs
NewQueueAnalyzer({MaxBatchSize b, MaxQueueSize 10 b, alpha, beta, gamma, delta of (model, a)}, {in, out})
.Size({TTFT, ITL, TPS of the server}); a record whose Size succeeds gets max_arrv_rate_per_replica =
float32(metrics.Throughput / 1000), every other field is kept.
"""
import numpy as np

from sweep_pair_ref import copy_records

F = np.float32


def size_inputs(wva, img, feasible):
    """the wva_queue_config / target rows of the records flagged in `feasible`, batch sizes left to the caller:
    {alpha, beta, gamma, delta of (model, a), in, out} and the server's {TTFT, ITL, TPS}
    -> (record indices gi, cfgs [n], targets [n, 3])"""
    gi = np.flatnonzero(feasible)
    s, a = gi // img.A, gi % img.A
    pi = img.srv_model[s].astype(np.int64) * img.A + a
    cfgs = np.zeros(len(gi), dtype=wva.abi.QUEUE_CONFIG_DTYPE)
    for name, arr in (("alpha", img.perf_alpha), ("beta", img.perf_beta), ("gamma", img.perf_gamma), ("delta", img.perf_delta)):
        cfgs[name] = arr[pi]
    cfgs["avg_input_tokens"] = img.srv_in_tokens[s]
    cfgs["avg_output_tokens"] = img.srv_out_tokens[s]
    targets = np.stack([img.srv_slo_ttft[s], img.srv_slo_itl[s], img.srv_slo_tps[s]], axis=1).astype(F)
    return gi, cfgs, targets


def sized_records(wva, oracle, img, recs, feasible, threads=1):
    """What wva_grid_pairs_size makes of the records (recs, feasible) of servers the records cover: the oracle's
    queue_size (QueueAnalyzer.Size) per record at its batch size b -> (sized copy of recs, status[S*A]) with status
    0 = no record, 1 = sized (max_arrv_rate_per_replica = float32(throughput / 1000)), 2 = Size error (unchanged)."""
    from concurrent.futures import ThreadPoolExecutor
    gi, cfgs, targets = size_inputs(wva, img, feasible)
    b = recs.batch_size[gi]
    cfgs["max_batch_size"] = b
    cfgs["max_queue_size"] = b * wva.abi.MAX_QUEUE_TO_BATCH_RATIO
    n = len(gi)
    tput = np.zeros(n, dtype=F)
    err = np.zeros(n, dtype=np.uint8)
    chunks = [slice(i, min(n, i + 64)) for i in range(0, n, 64)]

    def run(c):
        _, m, _, st = oracle.queue_size(cfgs[c], targets[c])   # ctypes drops the GIL: chunks run in parallel
        tput[c] = m["throughput"]
        err[c] = st

    with ThreadPoolExecutor(max(1, threads)) as ex:
        list(ex.map(run, chunks))
    out, _ = copy_records(wva, recs, feasible)
    status = np.zeros(len(feasible), dtype=np.uint8)
    ok = err == 0
    out.max_arrv_rate_per_replica[gi[ok]] = (tput[ok] / F(1000)).astype(F)
    status[gi] = np.where(ok, 1, 2)
    return out, status
