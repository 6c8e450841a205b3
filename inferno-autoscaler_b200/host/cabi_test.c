/* cabi_test.c — the C-ABI seen from plain C99, the way a cgo preamble sees it.
 *
 * (1) include/wva_b200.h compiles as C (cgo compiles the preamble with the C compiler, not C++);
 * (2) struct layouts are the natural-alignment ones cgo mirrors into Go (every field at a multiple of
 *     its size, no packing pragmas): offsets are asserted so that a change of the header that would
 *     silently change the Go-side layout fails here;
 * (3) on a box with a B200: the *_arrays entry points (what go/internal/native calls -- no struct of
 *     pointers crosses the boundary) give the same bytes as the struct forms, for the pair records and for
 *     the sweep's per-pair winners (wva_grid_pairs_fetch, wva_solve_grid) and for the load scenarios
 *     (wva_analyze_scenarios, wva_scenario_pairs_fetch); wva_grid_pairs_size flags every sweep record and
 *     nothing else.
 * Exit code 0 = ok (prints "no device" and stops after (2) when CUDA is unavailable). */
#include <stddef.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include "wva_b200.h"

#define CHECK(c) do { if (!(c)) { fprintf(stderr, "FAIL %s:%d: %s\n", __FILE__, __LINE__, #c); return 1; } } while (0)

_Static_assert(sizeof(wva_metrics) == 32, "wva_metrics");
_Static_assert(sizeof(wva_grid_best) == 32, "wva_grid_best");
_Static_assert(sizeof(wva_queue_config) == 32, "wva_queue_config");
_Static_assert(sizeof(wva_optimizer_spec) == 12, "wva_optimizer_spec");
_Static_assert(offsetof(wva_system_soa, acc_cost) == 16, "4 x int32 header, then pointers");
_Static_assert(sizeof(wva_system_soa) == 16 + 27 * sizeof(void*), "27 array pointers");
_Static_assert(offsetof(wva_system_soa, srv_cur_cost) == 16 + 26 * sizeof(void*), "last pointer");
_Static_assert(sizeof(wva_alloc_soa) == 9 * sizeof(void*), "9 array pointers");
_Static_assert(offsetof(wva_alloc_soa, max_arrv_rate_per_replica) == 8 * sizeof(void*), "last pointer");
_Static_assert(WVA_COMM_ID_BYTES == 128, "ncclUniqueId");

enum { S = 6, A = 3, M = 6, T = 2 };

int main(void) {
    CHECK(wva_abi_version() == WVA_ABI_VERSION);
    wva_ctx* ctx = NULL;
    int rc = wva_ctx_create(0, &ctx);
    if (rc != WVA_OK) {
        CHECK(rc == WVA_ECUDA && ctx == NULL && strlen(wva_last_error(NULL)) > 0);   /* fails loudly, no CPU fallback */
        printf("cabi_test: layout ok; no device (%s)\n", wva_last_error(NULL));
        return 0;
    }
    /* a tiny system, every array a separate allocation (as Go slices are) */
    float acc_cost[A] = {40.0f, 75.5f, 110.0f}; int32_t acc_mult[A] = {1, 2, 1}, acc_type[A] = {0, 1, 0};
    int64_t cap[T] = {0, 0};
    float al[M * A], be[M * A], ga[M * A], de[M * A]; int32_t mb[M * A], at[M * A], ac[M * A]; uint8_t pv[M * A];
    for (int i = 0; i < M * A; ++i) {
        al[i] = 6.0f + (float)(i % 7); be[i] = 0.05f + 0.03f * (float)(i % 5); ga[i] = 20.0f + 9.0f * (float)(i % 4);
        de[i] = 0.001f * (float)(1 + i % 3); mb[i] = 16 + 8 * (i % 5); at[i] = 256; ac[i] = 1 + (i % 2); pv[i] = 1;
    }
    int32_t sm[S], sin[S], sout[S], spr[S], smr[S], smb[S], sca[S], scr[S]; uint8_t stv[S], ska[S];
    float sar[S], stt[S], sit[S], stp[S], scc[S];
    for (int s = 0; s < S; ++s) {
        sm[s] = s; sar[s] = 30.0f * (float)(s + 1) * (float)(s + 1); sin[s] = 128 * (s + 1); sout[s] = 64 + 32 * s;
        stt[s] = 1000.0f; sit[s] = 80.0f; stp[s] = 0.0f; stv[s] = 1; spr[s] = 1 + s; smr[s] = s & 1; smb[s] = 0; ska[s] = 0;
        sca[s] = (s % 3 == 0) ? WVA_ACC_NONE : (s % A); scr[s] = (s % 3 == 0) ? 0 : 2; scc[s] = (s % 3 == 0) ? 0.0f : 150.0f;
    }
    sar[4] = 0.0f;   /* a zero-load server */
    CHECK(wva_system_upload_arrays(ctx, S, A, M, T, acc_cost, acc_mult, acc_type, cap, al, be, ga, de, mb, at, ac, pv, sm, sar, sin, sout,
                                   stt, sit, stp, stv, spr, smr, smb, ska, sca, scr, scc) == WVA_OK);
    int32_t acc1[S * A]; int64_t rep1[S * A], bat1[S * A]; float f1[6][S * A]; uint8_t fe1[S * A];
    CHECK(wva_analyze_pairs_arrays(ctx, acc1, rep1, bat1, f1[0], f1[1], f1[2], f1[3], f1[4], f1[5], fe1) == WVA_OK);
    int32_t key1[S], cacc1[S]; int64_t crep1[S], cbat1[S]; float cf1[6][S];
    CHECK(wva_solve_arrays(ctx, 1, 0, WVA_POLICY_NONE, key1, cacc1, crep1, cbat1, cf1[0], cf1[1], cf1[2], cf1[3], cf1[4], cf1[5]) == WVA_OK);

    /* the struct forms on the same inputs */
    wva_system_soa h;
    h.n_servers = S; h.n_accels = A; h.n_models = M; h.n_types = T;
    h.acc_cost = acc_cost; h.acc_multiplicity = acc_mult; h.acc_type = acc_type; h.type_capacity = cap;
    h.perf_alpha = al; h.perf_beta = be; h.perf_gamma = ga; h.perf_delta = de; h.perf_max_batch = mb; h.perf_at_tokens = at;
    h.perf_acc_count = ac; h.perf_valid = pv; h.srv_model = sm; h.srv_arrival_rpm = sar; h.srv_in_tokens = sin; h.srv_out_tokens = sout;
    h.srv_slo_ttft = stt; h.srv_slo_itl = sit; h.srv_slo_tps = stp; h.srv_target_valid = stv; h.srv_priority = spr;
    h.srv_min_replicas = smr; h.srv_max_batch = smb; h.srv_keep_acc = ska; h.srv_cur_acc = sca; h.srv_cur_replicas = scr; h.srv_cur_cost = scc;
    CHECK(wva_system_upload(ctx, &h) == WVA_OK);
    int32_t acc2[S * A]; int64_t rep2[S * A], bat2[S * A]; float f2[6][S * A]; uint8_t fe2[S * A];
    wva_alloc_soa o2 = {acc2, rep2, bat2, f2[0], f2[1], f2[2], f2[3], f2[4], f2[5]};
    CHECK(wva_analyze_pairs(ctx, &o2, fe2) == WVA_OK);
    int32_t key2[S], cacc2[S]; int64_t crep2[S], cbat2[S]; float cf2[6][S];
    wva_alloc_soa c2 = {cacc2, crep2, cbat2, cf2[0], cf2[1], cf2[2], cf2[3], cf2[4], cf2[5]};
    wva_optimizer_spec spec = {1, 0, WVA_POLICY_NONE};
    CHECK(wva_solve(ctx, &spec, key2, &c2) == WVA_OK);
    CHECK(!memcmp(acc1, acc2, sizeof acc1) && !memcmp(rep1, rep2, sizeof rep1) && !memcmp(bat1, bat2, sizeof bat1));
    CHECK(!memcmp(f1, f2, sizeof f1) && !memcmp(fe1, fe2, sizeof fe1));
    CHECK(!memcmp(key1, key2, sizeof key1) && !memcmp(cacc1, cacc2, sizeof cacc1) && !memcmp(crep1, crep2, sizeof crep1) && !memcmp(cf1, cf2, sizeof cf1));
    int nfe = 0; for (int i = 0; i < S * A; ++i) nfe += fe1[i];
    CHECK(nfe > 0);
    int64_t cnt[T]; float cst[T];
    CHECK(wva_allocate_by_type(ctx, cnt, cst) == WVA_OK);

    /* the sweep's per-pair winners: fetch and solve, arrays forms against struct forms */
    CHECK(wva_grid_set_pair_winners(ctx, 1) == WVA_OK);
    CHECK(wva_analyze_grid_device(ctx, 8, 32, 0) == WVA_OK);
    int32_t gacc1[S * A]; int64_t grep1[S * A], gbat1[S * A]; float gf1[6][S * A]; uint8_t gfe1[S * A];
    int32_t gacc2[S * A]; int64_t grep2[S * A], gbat2[S * A]; float gf2[6][S * A]; uint8_t gfe2[S * A];
    CHECK(wva_grid_pairs_fetch_arrays(ctx, gacc1, grep1, gbat1, gf1[0], gf1[1], gf1[2], gf1[3], gf1[4], gf1[5], gfe1) == WVA_OK);
    wva_alloc_soa g2 = {gacc2, grep2, gbat2, gf2[0], gf2[1], gf2[2], gf2[3], gf2[4], gf2[5]};
    CHECK(wva_grid_pairs_fetch(ctx, &g2, gfe2) == WVA_OK);
    CHECK(!memcmp(gacc1, gacc2, sizeof gacc1) && !memcmp(grep1, grep2, sizeof grep1) && !memcmp(gbat1, gbat2, sizeof gbat1));
    CHECK(!memcmp(gf1, gf2, sizeof gf1) && !memcmp(gfe1, gfe2, sizeof gfe1));
    int ngfe = 0; for (int i = 0; i < S * A; ++i) ngfe += gfe1[i];
    CHECK(ngfe > 0);
    CHECK(wva_solve_grid_arrays(ctx, 1, 0, WVA_POLICY_NONE, key1, cacc1, crep1, cbat1, cf1[0], cf1[1], cf1[2], cf1[3], cf1[4], cf1[5]) == WVA_OK);
    CHECK(wva_solve_grid(ctx, &spec, key2, &c2) == WVA_OK);
    CHECK(!memcmp(key1, key2, sizeof key1) && !memcmp(cacc1, cacc2, sizeof cacc1) && !memcmp(crep1, crep2, sizeof crep1) && !memcmp(cf1, cf2, sizeof cf1));
    /* Size on the records: a status byte for every record (1 sized / 2 Size failed), 0 where there is none */
    uint8_t gst[S * A];
    memset(gst, 0xee, sizeof gst);
    CHECK(wva_grid_pairs_size(ctx, gst) == WVA_OK);
    for (int i = 0; i < S * A; ++i) CHECK(gfe1[i] ? (gst[i] == 1 || gst[i] == 2) : gst[i] == 0);
    CHECK(wva_grid_set_pair_winners(ctx, 0) == WVA_OK);
    CHECK(wva_analyze_grid_device(ctx, 8, 32, 0) == WVA_OK);
    CHECK(wva_solve_grid(ctx, &spec, key2, &c2) == WVA_ESTATE);                 /* a sweep with the option off */
    CHECK(wva_grid_pairs_size(ctx, gst) == WVA_ESTATE);
    /* load scenarios (the image's rates, none, twice the image's): arrays forms against struct forms */
    enum { L = 3 };
    float lr[L * S];
    for (int i = 0; i < S; ++i) { lr[i] = sar[i]; lr[S + i] = 0.0f; lr[2 * S + i] = 2.0f * sar[i]; }
    int32_t lkey1[L * S], lacc1[L * S], lkey2[L * S], lacc2[L * S]; int64_t lrep1[L * S], lbat1[L * S], lrep2[L * S], lbat2[L * S];
    float lf1[6][L * S], lf2[6][L * S]; int64_t lcnt1[L * T], lcnt2[L * T]; float lcst1[L * T], lcst2[L * T];
    CHECK(wva_analyze_scenarios_arrays(ctx, L, lr, lkey1, lacc1, lrep1, lbat1, lf1[0], lf1[1], lf1[2], lf1[3], lf1[4], lf1[5], lcnt1, lcst1) == WVA_OK);
    CHECK(wva_scenario_pairs_fetch_arrays(ctx, 2, gacc1, grep1, gbat1, gf1[0], gf1[1], gf1[2], gf1[3], gf1[4], gf1[5], gfe1) == WVA_OK);
    wva_alloc_soa l2 = {lacc2, lrep2, lbat2, lf2[0], lf2[1], lf2[2], lf2[3], lf2[4], lf2[5]};
    CHECK(wva_analyze_scenarios(ctx, L, lr, lkey2, &l2, lcnt2, lcst2) == WVA_OK);
    CHECK(wva_scenario_pairs_fetch(ctx, 2, &g2, gfe2) == WVA_OK);
    CHECK(!memcmp(lkey1, lkey2, sizeof lkey1) && !memcmp(lacc1, lacc2, sizeof lacc1) && !memcmp(lrep1, lrep2, sizeof lrep1));
    CHECK(!memcmp(lbat1, lbat2, sizeof lbat1) && !memcmp(lf1, lf2, sizeof lf1) && !memcmp(lcnt1, lcnt2, sizeof lcnt1) && !memcmp(lcst1, lcst2, sizeof lcst1));
    CHECK(!memcmp(gacc1, gacc2, sizeof gacc1) && !memcmp(grep1, grep2, sizeof grep1) && !memcmp(gbat1, gbat2, sizeof gbat1));
    CHECK(!memcmp(gf1, gf2, sizeof gf1) && !memcmp(gfe1, gfe2, sizeof gfe1));
    CHECK(wva_analyze_scenarios(ctx, 0, lr, NULL, NULL, NULL, NULL) == WVA_EINVAL);
    CHECK(wva_scenario_pairs_fetch(ctx, L, &g2, gfe2) == WVA_EINVAL);
    printf("cabi_test: ok (%d feasible pairs, %d feasible sweep pairs, type counts %lld %lld)\n", nfe, ngfe, (long long)cnt[0], (long long)cnt[1]);
    wva_ctx_destroy(ctx);
    return 0;
}
