// wva_grid_scan.cuh — the candidate sweep with ONE WARP PER ROW and a PARALLEL ramp (k_grid_scan).
//
// A row is (server, accelerator, replicas): all its candidates share lambda, and the chain of batch size
// b is a prefix of the chain of b+1, so one ramp p[1..B] serves the whole row (as in k_grid_rows).  Here the
// 32 lanes of a warp hold 32 CONSECUTIVE batch sizes of the same row:
//
//   * the ramp is not stepped sequentially: lane l forms the ratio lambda/s[n] of its own state and the warp
//     builds p[n] = prod ratio, sum_{i<=n} p[i] and sum_{i<=n} i p[i] with three inclusive scans (5 shuffle
//     steps each) plus a carry from the previous 32 states.  ~20 FP64 instructions per lane and chunk
//     instead of 32 dependent ramp steps;
//   * every lane then evaluates its own candidate from (p[b], sum, sum i p) with the certified closed-form
//     tail (cert_eval_fast: two reciprocals instead of eight IEEE divisions);
//   * the 32 results of a chunk are 1 KB of contiguous cube: one fully coalesced store per float4 half
//     (k_grid_rows writes 32 B per lane at a 16 KB stride);
//   * lanes of a warp share the replica count, so the "rate > RateRange.Max" early-outs and the died-out
//     tail are (nearly) warp-uniform.
//
// Exactness.  The scans reassociate the ramp, so the ramp values are NOT bit-identical to the reference's
// sequential p[n] (those of k_grid_rows are).  They do not have to be: the certificate (DESIGN.md 4.iii)
// never used bit-identity of the ramp, only a bound on the distance between the quantities we feed into the
// float32 roundings and their exact-arithmetic values.  Error budget of this kernel, in units of u = 2^-53,
// relative, for candidate b (N = b, K = 11 b):
//     ratio_i = lambda * rcp(s_i)                 <= 2 u     (rcp_refined is within 1 ulp of 1/s_i)
//     p[n]   = product of n ratios, n-1 roundings <= 3 n u
//     sums   : positive terms, scan depth 5 + one carry addition per chunk <= (5 + n/32 + 1) u on top
//     tail   : closed forms with two reciprocals  <= 128 u   (see cert_eval_fast)
// i.e. <= (3.1 N + 140) u <= 0.3 K u + 140 u on every aggregate, against the reference's own <= 8 K u distance
// from exact arithmetic.  The acceptance test uses E = 64 K u >= 8 K u + 0.3 K u + 140 u for every K >= 3
// (K >= 11 here), so an accepted float32 is the reference's float32; an ambiguous one goes to the exact-chain
// kernels exactly as before.  The parity tests compare the ENTIRE config-2 cube and >= 1e6 candidates of
// configs 3-5 (+ every deferred candidate, + exhaustive winner proofs) with the oracle.
//
// A lane whose p leaves the value window [2^-800, 2^990) on the high side (or is NaN) makes the rest of the
// row "broken": those candidates go to the exact-chain kernels.  Leaving it on the low side with the ratio
// already <= 0.998 (tame table: ratios do not grow again) means the chain has died out: p := 0, which is
// within the budget above since sum >= 1.
#pragma once

namespace wva {

// 1/x for a positive normal x well inside the exponent range: MUFU seed + two Newton steps (<= 1 ulp)
__device__ __forceinline__ double rcp_pos(double x) { return rcp_refined(x); }

// The certificate of cert_eval with the divisions folded into two reciprocals.  yTail = rcp_refined(sTail).
// Own error (relative, units of u): oneR, r <= 2; inv <= 4; T0 <= 7, T1 <= 11 (+ the exp/log1p term of cert_eval when
// x < 140: <= 80 on 1 - r^M (1 + x)); S, U <= 100; invS <= 102; every aggregate <= 128.
__device__ __noinline__ bool cert_eval_fast(const double pN, const double sumRamp, const double uN, const double lam,
                                               const double sTail, const double yTail, const int N, const int K,
                                               const float lambda, SolveStats& o) {
    const int M = K - N;
    if (M < 1 || K > (1 << 20)) return false;
    const double oneR = (sTail - lam) * yTail;                 // 1 - r: exact subtraction of two float32 values
    if (!(oneR >= 0x1p-11) || !(oneR < 1.0)) return false;      // r in (0, 0.9995]
    const double r = lam * yTail;
    const double x = (double)M * oneR;
    if (!(x >= 0.3)) return false;
    const double inv = rcp_pos(oneR);
    double T0 = r * inv;
    double T1 = T0 * inv;
    double rM = 0.0;
    if (x < 140.0) {                                            // r^M <= exp(-x): below 2^-200 it cannot matter
        rM = exp((double)M * log1p(-oneR));
        T0 = T0 * (1.0 - rM);
        T1 = T1 * (1.0 - rM * (1.0 + x));
    }
    const double pT0 = pN * T0;
    const double S = sumRamp + pT0;
    const double U = uN + (pN * T1 + (double)N * pT0);
    if (!(S < 0x1p1000) || !(U < 0x1p1000) || !(S > 0x1p-1000)) return false;
    const double invS = rcp_pos(S);
    const double tailMass = pT0 * invS;                          // 1 - sumP at i = N, without cancellation
    const double pK = (pN * rM) * invS;
    const double inSys = U * invS;
    const double inServ = uN * invS + tailMass * (double)N;
    const double Ku = (double)K * 0x1p-53;
    const double E = 64.0 * Ku;
    float inSysF, inServF, pKlo;
    if (!same_f32(inSys, E * inSys, inSysF)) return false;
    if (!same_f32(inServ, E * inServ + 4.0 * Ku * (double)N, inServF)) return false;
    if (!same_f32(pK, 2.0 * E * pK, pKlo)) {
        const float a = 1.0f - (float)(pK * (1.0 - 2.0 * E)), b = 1.0f - (float)(pK * (1.0 + 2.0 * E));
        if (a != b) return false;
        finish_stats_f32(o, lambda, inServF, inSysF, a);
    } else {
        finish_stats_f32(o, lambda, inServF, inSysF, 1.0f - pKlo);
    }
    o.rho = 0.0f;     // model.rho only feeds the stale-rho validity test, vacuous for K >= 2
    return true;
}

__device__ __forceinline__ double shfl_up_d(double v, int o) { return __shfl_up_sync(0xffffffffu, v, o); }

// Per-row result of the exact sequential ramp (phase A).  A lightly loaded row's chain dies out after a few
// states; from there on the reference's sums no longer change and 1 - sumP is pure rounding noise of ITS
// summation order, which no tolerance-based certificate can reproduce -- those candidates need the exact
// sequential arithmetic (the "stopped" path of k_grid_rows, same rule, same code shape):
//   stopB   first batch size whose candidates use the frozen exact sums (INT_MAX: the row never stops)
//   brokenB first batch size from which the row must go to the exact-chain kernels (window exit in the exact ramp)
struct ScanRow { int stopB, brokenB; double exInSys, exSumP; int nGood, pad; };   // nGood: table entries [0, nGood) are usable (pair-wide)

// The exact ramp of one row up to its stop: the reference's recurrence, sequential, bit-identical
// (mm1modelstatedependent.go:77-112), with solve_stream's truncation rule at a 2^10 stricter threshold.
__device__ __noinline__ void scan_row_exact(const double* rateD, const double* rcp, const float* rateF, const int B, const int nGood,
                                               const bool tame, const float lambda, ScanRow& out, unsigned long long& steps) {
    out.stopB = 0x7fffffff; out.brokenB = 0x7fffffff; out.exInSys = 0.0; out.exSumP = 0.0; out.nGood = nGood; out.pad = 0;
    const double lam = (double)lambda;
    if (!(lam >= 0x1p-100 && lam <= 0x1p20)) { out.brokenB = 1; return; }
    // a row stops only after its ratios have dropped under 0.998: with a tame (non-decreasing) table that never
    // happens when even the largest rate is too small
    if (!tame || !(lambda <= 0.998f * rateF[(nGood < B ? nGood : B) - 1 < 0 ? 0 : (nGood < B ? nGood : B) - 1])) return;
    double p = 1.0, sum = 1.0;
    unsigned thrHi = 0u, hmin = 0x3ff00000u;
    const int nEnd = nGood < B ? nGood : B;
    for (int n = 0; n < nEnd; ++n) {
        const double pn = div_core(p * lam, rateD[n], rcp[n]);
        const unsigned hq = (unsigned)__double2hiint(pn);
        if (hq - WVA_WIN_LO >= WVA_WIN_SPAN) { out.brokenB = n + 1; break; }
        sum += pn; p = pn;
        ++steps;
        if (n == 0 && pn >= 0x1p-400) thrHi = (unsigned)__double2hiint((0x1p-68 * fmin(1.0, pn)) / (double)(11 * B));
        hmin = hq < hmin ? hq : hmin;
        if (hq < thrHi && lambda <= 0.998f * rateF[n] && sum <= 0x1p400) {
            const int b = n + 1;
            const double S = sum;
            if ((int)(hmin >> 20) - (int)((unsigned)__double2hiint(S) >> 20) < -1000) { out.brokenB = b; break; }
            const double yS = rcp_refined(S);
            double q = div_core(1.0, S, yS), pp = 1.0, di = 0.0, exSumP = q, exInSys = 0.0;
            for (int i = 1; i <= b; ++i) {
                pp = div_core(pp * lam, rateD[i - 1], rcp[i - 1]);
                q = div_core(pp, S, yS);
                di += 1.0;
                exInSys += di * q;
                exSumP += q;
            }
            steps += (unsigned long long)b;
            out.stopB = b; out.exInSys = exInSys; out.exSumP = exSumP;
            break;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// The sweep as three kernels, so that each gets the register allocation (and occupancy) its work needs:
//
//   k_scan_prep   block = (pair, chunk of rows), one THREAD per row: builds the pair's {rate, reciprocal} table
//                 (published in gp.pair_tab for the other kernels), runs the exact ramp of every row to its stop
//                 (scan_row_exact) and leaves one ScanRow per row in gp.row_info; fills the status / cube of pairs
//                 whose lookups fail.
//   k_scan_cert   one WARP per row, the batch sizes BEFORE the row's stop: ramp by warp scans + cert_eval_fast
//                 (FP64-heavy, ~100 registers).
//   k_scan_lean   one WARP per row, the batch sizes FROM the row's stop on: the reference's sums are frozen there,
//                 a candidate is a dozen float32 operations and a 33-byte store (few registers, high occupancy;
//                 bound by the cube's HBM write).  In the synthetic sets ~13 of a row's 16 chunks are of this kind.
// k_scan_cert and k_scan_lean write disjoint candidates; a 32-candidate chunk that contains the stop belongs to
// k_scan_cert entirely.
// ---------------------------------------------------------------------------------------------------------------
#define WVA_SCAN_WARPS 8
#define WVA_SCAN_MAXROWS 64        /* rows (replica counts) per block */

struct ScanBlock {                 // what every kernel derives from blockIdx
    int pairSlice, rBeg, rEnd, pairLocal, sl, a, s;
};
__device__ __forceinline__ ScanBlock scan_block(const DevSystem& sys, const GridParams& gp) {
    ScanBlock k;
    k.pairSlice = blockIdx.x / gp.n_rchunks;
    const int rchunk = blockIdx.x % gp.n_rchunks;
    k.rBeg = rchunk * gp.r_chunk + 1;
    k.rEnd = (k.rBeg + gp.r_chunk - 1 < gp.r_max) ? k.rBeg + gp.r_chunk - 1 : gp.r_max;
    k.pairLocal = gp.pair_base + k.pairSlice;
    k.sl = k.pairLocal / sys.A; k.a = k.pairLocal % sys.A;
    k.s = gp.s0 + k.sl;
    return k;
}
// pair usable for the sweep?  (status of all its candidates otherwise)
__device__ __forceinline__ int scan_pair_status(const DevSystem& sys, int s, int a, GridServer& gs) {
    if (!(pair_lookups_ok(sys, s, a) && is_candidate_accel(sys, s, a))) return WVA_CAND_ERR_PAIR;
    load_grid_server(sys, s, a, gs);
    if (gs.inTok < 0 || gs.outTok < 1 || gs.sloTTFT < 0.0f || gs.sloITL < 0.0f || gs.sloTPS < 0.0f) return WVA_CAND_ERR_CONFIG;
    return WVA_CAND_OK;
}

__global__ void __launch_bounds__(WVA_SCAN_MAXROWS)
k_scan_prep(DevSystem sys, GridParams gp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* rateD = reinterpret_cast<double*>(smem_raw);
    double* rcp = rateD + gp.b_max;
    float* rateF = reinterpret_cast<float*>(rcp + gp.b_max);
    __shared__ int sh_nGood;
    const ScanBlock k = scan_block(sys, gp);
    const int B = gp.b_max, R = gp.r_max;
    if (threadIdx.x == 0) sh_nGood = B;
    GridServer gs;
    const int blockStatus = scan_pair_status(sys, k.s, k.a, gs);
    const size_t candBase = ((size_t)k.pairLocal * R) * (size_t)B;
    ScanRow* rowInfo = gp.row_info + (size_t)k.pairSlice * R;
    if (blockStatus != WVA_CAND_OK) {
        const size_t n = (size_t)(k.rEnd - k.rBeg + 1) * B, off = (size_t)(k.rBeg - 1) * B;
        if (gp.cube) {
            float4* c = reinterpret_cast<float4*>(&gp.cube[candBase + off]);
            const float4 z = make_float4(0, 0, 0, 0);
            for (size_t j = threadIdx.x; j < 2 * n; j += blockDim.x) c[j] = z;
        }
        if (gp.status) for (size_t j = threadIdx.x; j < n; j += blockDim.x) gp.status[candBase + off + j] = (unsigned char)blockStatus;
        for (int rr = threadIdx.x; rr <= k.rEnd - k.rBeg; rr += blockDim.x) { ScanRow row; row.stopB = row.brokenB = -1; row.exInSys = row.exSumP = 0.0; row.nGood = 0; row.pad = 0; rowInfo[k.rBeg - 1 + rr] = row; }
        return;
    }
    __syncthreads();
    ServFormula sf; sf.init(gs.sp, gs.inTok, gs.outTok);
    double2* gtab = gp.pair_tab + (size_t)k.pairSlice * B;
    for (int i = threadIdx.x; i < B; i += blockDim.x) {
        const float rt = sf.rate(i + 1);
        rateF[i] = rt;
        const double d = (double)rt;
        const double y = rcp_refined(d);
        rateD[i] = d; rcp[i] = y;
        if (k.rBeg == 1) {                                       // one block per pair publishes the tables
            gtab[i] = make_double2(d, y);
            // RateRange.Max (queueanalyzer.go:116-118) and RateTargetTPS (:231-234, :246) of batch size i + 1
            const float rateMax = (rt * (1.0f - WVA_EPSILON)) * 1000.0f;
            gp.rate_tab[(size_t)k.pairSlice * B + i] = make_float2(rateMax, ((rateMax / 1000.0f) * (1.0f - WVA_STABILITY_SAFETY)) * 1000.0f);
        }
        if (!(rt > 0.0f) || !(rt < CUDART_INF_F)) atomicMin(&sh_nGood, i);
    }
    const bool tame = tame_parms(gs.sp, gs.inTok, gs.outTok);
    __syncthreads();
    const int nGood = sh_nGood;
    unsigned long long steps = 0;
    for (int rr = threadIdx.x; rr <= k.rEnd - k.rBeg; rr += blockDim.x) {
        const float lambdaA = (gs.totalRate / (float)(k.rBeg + rr)) / 1000.0f;
        ScanRow row;
        scan_row_exact(rateD, rcp, rateF, B, nGood, tame, lambdaA, row, steps);
        rowInfo[k.rBeg - 1 + rr] = row;
    }
    for (int o = 16; o > 0; o >>= 1) steps += __shfl_down_sync(0xffffffffu, steps, o);
    if ((threadIdx.x & 31) == 0 && steps) atomicAdd(&gp.counters[0], steps);
}

// Pair- and row-invariant parts of a candidate's float32 epilogue (QueueAnalyzer.Analyze after the Solve,
// queueanalyzer.go:152-173, EffectiveConcurrency :296-302): the divisors of the two divisions that do not depend on
// the batch size are inverted once (div_hoisted_f32: same instruction sequence as nvcc's `/`, reciprocal hoisted).
struct ScanPairCtx {
    float base, den, yDen, d1, gamma, alpha, beta; bool denOk, inZero;
    float sloTTFT, sloITL, sloTPS;
};
__device__ __forceinline__ ScanPairCtx scan_pair_ctx(const GridServer& gs) {
    ScanPairCtx pc;
    const float tokens = (float)(gs.outTok - 1);
    const float at = gs.sp.alpha * tokens;
    pc.base = gs.sp.gamma + at;
    pc.d1 = gs.sp.delta * (float)gs.inTok;
    const float d2 = gs.sp.beta * tokens;
    pc.den = pc.d1 + d2;
    pc.yDen = rcp_refined_f32(pc.den); pc.denOk = f32_div_window(pc.den);
    pc.gamma = gs.sp.gamma; pc.alpha = gs.sp.alpha; pc.beta = gs.sp.beta; pc.inZero = gs.inTok == 0;
    pc.sloTTFT = gs.sloTTFT; pc.sloITL = gs.sloITL; pc.sloTPS = gs.sloTPS;
    return pc;
}
struct ScanRowCtx {                // row constants
    float rate, lambda; unsigned long long rowKey; bool valueOk, repOk;
    wva_metrics* rowCube; unsigned char* rowStatus;
};
// one analysed candidate: metrics from (avgNumInServers, avgNumInSystem, throughput, avgRespTime, avgServTime, avgWaitTime),
// SLO tests, stores.  Returns feasible.  rateMax / rateTPS come from k_scan_prep's table.
__device__ __forceinline__ bool scan_finish(const ScanPairCtx& pc, const ScanRowCtx& rc, const SolveStats& so, const int n, const float bF,
                                            const float rateMax, const float rateTPS, float& itlOut, float& ttftOut, float& rhoOut) {
    const float num = so.avgServTime - pc.base;
    const float effN = div_hoisted_f32(num, pc.den, pc.yDen, pc.denOk);
    const float effConc = (effN > 0.0f && effN <= bF) ? effN : go_minf(go_maxf(effN, 0.0f), bF);      // the clamp only matters outside (0, N]
    float rho = div_hoisted_f32(so.avgNumInServers, bF, rcp_refined_f32(bF), true);                   // bF = float32(b), 1 <= b <= 8192
    if (!(rho > 0.0f && rho <= 1.0f)) rho = go_minf(go_maxf(rho, 0.0f), 1.0f);
    const float prefill = pc.inZero ? 0.0f : pc.gamma + pc.d1 * effConc;
    const float token = pc.alpha + pc.beta * effConc;
    const float ttft = so.avgWaitTime + prefill;
    const bool feasible = (!(pc.sloTTFT > 0.0f) || ttft <= pc.sloTTFT) && (!(pc.sloITL > 0.0f) || token <= pc.sloITL) &&
                          (!(pc.sloTPS > 0.0f) || rc.rate <= rateTPS) && rc.repOk;
    itlOut = token; ttftOut = ttft; rhoOut = rho;
    if (rc.rowCube) {
        float4* c = reinterpret_cast<float4*>(&rc.rowCube[n]);
        c[0] = make_float4(so.throughput * 1000.0f, so.avgRespTime, so.avgWaitTime, so.avgNumInServers);
        c[1] = make_float4(prefill, token, rateMax, rho);
    }
    if (rc.rowStatus) rc.rowStatus[n] = (unsigned char)(WVA_CAND_OK | (feasible ? WVA_CAND_FEASIBLE : 0));
    return feasible;
}
__device__ __forceinline__ void scan_store_error(const ScanRowCtx& rc, const int n, const int st) {
    if (rc.rowCube) {
        float4* c = reinterpret_cast<float4*>(&rc.rowCube[n]);
        const float4 z = make_float4(0, 0, 0, 0);
        c[0] = z; c[1] = z;
    }
    if (rc.rowStatus) rc.rowStatus[n] = (unsigned char)st;
}
__device__ __forceinline__ ScanRowCtx scan_row_ctx(const GridServer& gs, const GridParams& gp, const int a, const int r, const size_t candBase) {
    ScanRowCtx rc;
    rc.rate = gs.totalRate / (float)r;
    rc.lambda = rc.rate / 1000.0f;
    const float cost = gs.accCost * (float)go_muli(gs.numInst, (long long)r);
    float value = transition_penalty(gs.curAcc, gs.curRep, gs.curCost, a, (long long)r, cost);
    value = value + 0.0f;
    rc.valueOk = value == value;                               // a NaN value is never selected
    rc.rowKey = make_key(value, a, r, 1);
    rc.repOk = r >= gs.minReplicas;
    const size_t rowBase = candBase + (size_t)(r - 1) * gp.b_max;
    rc.rowCube = gp.cube ? gp.cube + rowBase : nullptr;
    rc.rowStatus = gp.status ? gp.status + rowBase : nullptr;
    return rc;
}
// Within a row the key grows with the batch size, so the row's best candidate is its FIRST feasible one: the warp keeps
// (first feasible n, its metrics) per row and compares rows once per row instead of once per candidate.
struct ScanBest { unsigned long long key; float itl, ttft, rho; };
__device__ __forceinline__ void scan_row_best(ScanBest& best, bool& rowHas, const ScanRowCtx& rc, const bool feasible, const int n,
                                              const float itl, const float ttft, const float rho) {
    if (rowHas) return;                                            // warp-uniform
    const unsigned m = __ballot_sync(0xffffffffu, feasible && rc.valueOk);
    if (!m) return;
    rowHas = true;
    const int src = __ffs(m) - 1;
    const int nWin = __shfl_sync(0xffffffffu, n, src);
    const float i_ = __shfl_sync(0xffffffffu, itl, src), t_ = __shfl_sync(0xffffffffu, ttft, src), r_ = __shfl_sync(0xffffffffu, rho, src);
    const unsigned long long key = rc.rowKey + (unsigned long long)nWin;
    if (key < best.key) { best.key = key; best.itl = i_; best.ttft = t_; best.rho = r_; }
}

// block argmin + counters (shared by k_scan_cert / k_scan_lean); slotBase separates the two kernels' slots
__device__ __forceinline__ void scan_block_reduce(const DevSystem& sys, const GridParams& gp, const GridServer& gs, const ScanBlock& k, const int slot,
                                                  unsigned long long bestKey, float bestItl, float bestTtft, float bestRho,
                                                  unsigned long long steps, unsigned long long algSteps, unsigned long long okCount,
                                                  unsigned long long* sh_key, unsigned long long* sh_cnt) {
    const int lane = threadIdx.x & 31;
    unsigned long long warpKey = bestKey;
    for (int o = 16; o > 0; o >>= 1) {
        const unsigned long long other = __shfl_down_sync(0xffffffffu, warpKey, o);
        if (other < warpKey) warpKey = other;
        steps += __shfl_down_sync(0xffffffffu, steps, o);
        algSteps += __shfl_down_sync(0xffffffffu, algSteps, o);
        okCount += __shfl_down_sync(0xffffffffu, okCount, o);
    }
    if (lane == 0) {
        if (warpKey != WVA_KEY_NONE) atomicMin(sh_key, warpKey);
        atomicAdd(&sh_cnt[0], steps); atomicAdd(&sh_cnt[1], algSteps); atomicAdd(&sh_cnt[2], okCount);
    }
    __syncthreads();
    const unsigned long long blockKey = *sh_key;
    if (blockKey != WVA_KEY_NONE && bestKey == blockKey) {
        GridSlot sl_; sl_.key = blockKey; sl_.itl = bestItl; sl_.ttft = bestTtft; sl_.rho = bestRho; sl_.sl = k.sl; sl_.pad = 0;
        const int r = (int)((blockKey >> 14) & 0x3ff) + 1;
        sl_.cost = gs.accCost * (float)go_muli(gs.numInst, (long long)r);
        gp.block_slot[slot] = sl_;
        atomicMin(&gp.keys[k.sl], blockKey);
        if (gp.pair_keys) atomicMin(&gp.pair_keys[gp.pair_base + (int)(blockIdx.x / (unsigned)gp.n_rchunks)], blockKey);   // a block covers one pair (index re-derived: no register live across the sweep)
    }
    if (threadIdx.x == 0) {
        atomicAdd(&gp.counters[0], sh_cnt[0]); atomicAdd(&gp.counters[1], sh_cnt[1]); atomicAdd(&gp.counters[2], sh_cnt[2]);
    }
}

// ---- the batch sizes from a row's stop on: frozen exact sums ----------------------------------------------------------
__global__ void __launch_bounds__(WVA_SCAN_WARPS * 32, 5)
k_scan_lean(DevSystem sys, GridParams gp) {
    __shared__ unsigned long long sh_key;
    __shared__ unsigned long long sh_cnt[3];
    const ScanBlock k = scan_block(sys, gp);
    const int B = gp.b_max, R = gp.r_max;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = gridDim.x + blockIdx.x;                       // second half of gp.block_slot
    __shared__ int sh_next;
    if (threadIdx.x == 0) { sh_key = WVA_KEY_NONE; sh_cnt[0] = sh_cnt[1] = sh_cnt[2] = 0; gp.block_slot[slot].key = WVA_KEY_NONE; sh_next = 0; }
    GridServer gs;
    if (scan_pair_status(sys, k.s, k.a, gs) != WVA_CAND_OK) return;       // k_scan_prep wrote the pair's status
    __syncthreads();
    const ScanPairCtx pc = scan_pair_ctx(gs);
    const size_t candBase = ((size_t)k.pairLocal * R) * (size_t)B;
    const float2* __restrict__ rtab = gp.rate_tab + (size_t)k.pairSlice * B;
    const ScanRow* __restrict__ rowInfo = gp.row_info + (size_t)k.pairSlice * R;
    ScanBest best; best.key = WVA_KEY_NONE; best.itl = best.ttft = best.rho = 0.0f;
    unsigned long long algSteps = 0, okCount = 0;
    // rows are handed out dynamically (a shared counter): their lengths differ by an order of magnitude
    for (;;) {
        int r = 0;
        if (lane == 0) r = k.rBeg + atomicAdd(&sh_next, 1);
        r = __shfl_sync(0xffffffffu, r, 0);
        if (r > k.rEnd) break;
        const ScanRow row = rowInfo[r - 1];
        if (row.stopB > B) continue;                                // the row never stops: all of it belongs to k_scan_cert
        const ScanRowCtx rc = scan_row_ctx(gs, gp, k.a, r, candBase);
        const float lambda = rc.lambda;
        const bool rowOk = rc.rate > 0.0f && !(lambda < 0.0f);
        const int rowErr = !(rc.rate > 0.0f) ? WVA_CAND_ERR_RATE_LE0 : WVA_CAND_ERR_MODEL;
        const double oneMinusSumP = 1.0 - row.exSumP;
        const float inSysF = (float)row.exInSys;
        const float tput = lambda * (1.0f - 0.0f);                  // throughput = lambda * (1 - float32(p[K])), p[K] rounds to 0
        const float respRow = inSysF / tput;                        // avgRespTime: the same for every stopped candidate of the row
        const float yT = rcp_refined_f32(tput); const bool tOk = f32_div_window(tput);
        // first chunk that lies entirely at or after the stop (the chunk containing the stop is k_scan_cert's)
        const int cFirst = ((row.stopB - 1 + 31) / 32) * 32;
        double bD = (double)(cFirst + lane + 1);
        float bF = (float)(cFirst + lane + 1);
        bool rowHas = false;
        unsigned okRow = 0, algRow = 0;
        float2 rmNext = (cFirst + lane < B) ? rtab[cFirst + lane] : make_float2(0.0f, 0.0f);     // one chunk ahead of its use
        for (int c0 = cFirst; c0 < B; c0 += 32, bD += 32.0, bF += 32.0f) {
            const int n = c0 + lane;
            const float2 rmCur = rmNext;
            if (n + 32 < B) rmNext = rtab[n + 32];
            bool feasible = false; float itl = 0.0f, ttft = 0.0f, rho = 0.0f;
            if (n < B) {
                if (n + 1 > row.nGood) {                           // bad table entry: the literal path decides (listed by k_scan_cert,
                                                                   // whose lists the host reads before this kernel has finished)
                } else {
                    const float2 rm = rmCur;
                    if (!rowOk) scan_store_error(rc, n, rowErr);
                    else if (rc.rate > rm.x) scan_store_error(rc, n, WVA_CAND_ERR_RATE_MAX);
                    else {
                        // exact: avgNumInServers is captured at i == b (mm1modelstatedependent.go:52-54) from sums that no longer
                        // change; float32(p[K]) < 2^-58 so throughput == lambda
                        SolveStats so;
                        const double inServ = row.exInSys + oneMinusSumP * bD;
                        so.avgNumInServers = (float)inServ;
                        so.avgNumInSystem = inSysF;
                        so.throughput = tput;
                        so.avgRespTime = respRow;
                        so.avgServTime = div_hoisted_f32(so.avgNumInServers, tput, yT, tOk);
                        so.avgWaitTime = so.avgRespTime - so.avgServTime;
                        if (so.avgWaitTime < 0.0f) so.avgWaitTime = 0.0f;
                        ++okRow; algRow += 22u * (unsigned)(n + 1) + 2u;
                        feasible = scan_finish(pc, rc, so, n, bF, rm.x, rm.y, itl, ttft, rho);
                    }
                }
            }
            scan_row_best(best, rowHas, rc, feasible, n, itl, ttft, rho);
        }
        okCount += okRow; algSteps += algRow;
    }
    scan_block_reduce(sys, gp, gs, k, slot, best.key, best.itl, best.ttft, best.rho, 0ULL, algSteps, okCount, &sh_key, sh_cnt);
}

// ---- the batch sizes before a row's stop: ramp by warp scans + certificate --------------------------------------------
// MINB: resident blocks per SM the register allocation targets (2: 124 registers, no spills; 3: 80 registers, 36 B of
// spills, 24 warps per SM) -- both are built, wva_set_certified_tails picks (results identical)
template <int MINB>
__global__ void __launch_bounds__(WVA_SCAN_WARPS * 32, MINB)
k_scan_cert(DevSystem sys, GridParams gp) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    double* rateD = reinterpret_cast<double*>(smem_raw);
    double* rcp = rateD + gp.b_max;
    float* rateF = reinterpret_cast<float*>(rcp + gp.b_max);
    __shared__ unsigned long long sh_key;
    __shared__ unsigned long long sh_cnt[3];
    __shared__ int sh_need, sh_next;
    const ScanBlock k = scan_block(sys, gp);
    const int B = gp.b_max, R = gp.r_max;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int slot = blockIdx.x;
    if (threadIdx.x == 0) { sh_key = WVA_KEY_NONE; sh_cnt[0] = sh_cnt[1] = sh_cnt[2] = 0; gp.block_slot[slot].key = WVA_KEY_NONE; sh_need = 0; sh_next = 0; }
    // the pair's constants live in shared memory: the main loop would otherwise carry ~30 registers of them
    __shared__ GridServer sh_gs;
    __shared__ ScanPairCtx sh_pc;
    __shared__ int sh_status;
    if (threadIdx.x == 0) {
        GridServer g0;
        sh_status = scan_pair_status(sys, k.s, k.a, g0);
        if (sh_status == WVA_CAND_OK) { sh_gs = g0; sh_pc = scan_pair_ctx(g0); }
    }
    __syncthreads();
    if (sh_status != WVA_CAND_OK) return;
    const GridServer& gs = sh_gs;
    const size_t candBase = ((size_t)k.pairLocal * R) * (size_t)B;
    const double2* __restrict__ gtab = gp.pair_tab + (size_t)k.pairSlice * B;
    const ScanRow* __restrict__ rowInfo = gp.row_info + (size_t)k.pairSlice * R;
    // candidates behind a bad table entry (rate not positive / not finite) in k_scan_lean's part of a row: listed here
    for (int r = k.rBeg + warp; r <= k.rEnd; r += WVA_SCAN_WARPS) {
        const ScanRow row = rowInfo[r - 1];
        if (row.nGood >= B || row.stopB > B) continue;
        const int cFirst = ((row.stopB - 1 + 31) / 32) * 32;
        for (int n = (cFirst > row.nGood ? cFirst : row.nGood) + lane; n < B; n += 32) {
            const int k0 = atomicAdd(gp.slow_count, 1);
            if (k0 < gp.slow_cap) gp.slow_list[k0] = (unsigned long long)(candBase + (size_t)(r - 1) * B + n);
        }
    }
    // how far this block's rows reach before their stops (the table is only needed up to there)
    int need = 0;
    for (int rr = threadIdx.x; rr <= k.rEnd - k.rBeg; rr += blockDim.x) {
        const ScanRow row = rowInfo[k.rBeg - 1 + rr];
        const int lim = row.stopB > B ? B : ((row.stopB - 1 + 31) / 32) * 32;
        need = need > lim ? need : lim;
    }
    if (need) atomicMax(&sh_need, need);
    __syncthreads();
    need = sh_need < B ? sh_need : B;
    if (need == 0) return;                                          // every row of the block stops in its first chunk... and k_scan_lean has it
    for (int i = threadIdx.x; i < need; i += blockDim.x) {
        const double2 v = gtab[i];
        rateD[i] = v.x; rcp[i] = v.y; rateF[i] = (float)v.x;
    }
    const bool tame = tame_parms(gs.sp, gs.inTok, gs.outTok);
    __syncthreads();

    const ScanPairCtx& pc = sh_pc;
    const float2* __restrict__ rtab = gp.rate_tab + (size_t)k.pairSlice * B;
    ScanBest best; best.key = WVA_KEY_NONE; best.itl = best.ttft = best.rho = 0.0f;
    unsigned long long steps = 0, algSteps = 0, okCount = 0;
    for (;;) {
        int r = 0;
        if (lane == 0) r = k.rBeg + atomicAdd(&sh_next, 1);         // rows handed out dynamically: 1 to 16 chunks each
        r = __shfl_sync(0xffffffffu, r, 0);
        if (r > k.rEnd) break;
        const ScanRow row = rowInfo[r - 1];
        const int cEnd = row.stopB > B ? B : ((row.stopB - 1 + 31) / 32) * 32;       // chunks [0, cEnd) are this kernel's
        if (cEnd == 0) continue;
        bool rowHas = false;
        float2 rmNext = (lane < B) ? rtab[lane] : make_float2(0.0f, 0.0f);            // one chunk ahead of its use
        const ScanRowCtx rc = scan_row_ctx(gs, gp, k.a, r, candBase);
        const float lambda = rc.lambda;
        const double lam = (double)lambda;
        const bool rateOk = rc.rate > 0.0f;
        const size_t rowBase = candBase + (size_t)(r - 1) * B;
        const double oneMinusSumP = 1.0 - row.exSumP;
        // carries of the three scans: state 0 is p = 1, sum = 1, sum i p = 0
        double carryP = 1.0, carrySum = 1.0, carryU = 0.0;
        bool rowBroken = false;        // the scan ramp left the value window: later candidates need the exact chain
        for (int c0 = 0; c0 < cEnd; c0 += 32) {
            const int n = c0 + lane, b = n + 1;
            const bool inRow = n < B;
            const float2 rm = rmNext;
            if (n + 32 < B) rmNext = rtab[n + 32];
            const bool stoppedLane = b >= row.stopB;
            double p = 0.0, sum = 0.0, uN = 0.0;
            bool broken = rowBroken || !inRow || b >= row.brokenB || b > row.nGood;
            if (c0 + 1 < row.brokenB && !rowBroken) {              // warp-uniform
                // ---- ramp states c0+1 .. c0+32 by scans --------------------------------------------------------
                double P = (inRow && b <= row.nGood) ? lam * rcp[n] : 1.0;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) { const double t = shfl_up_d(P, o); if (lane >= o) P *= t; }
                p = carryP * P;
                const unsigned hq = (unsigned)__double2hiint(p);
                bool laneBroken = false;
                if (hq - WVA_WIN_LO >= WVA_WIN_SPAN) {
                    // below the window (0 and subnormals included) after the ratios have dropped under 0.998: died out
                    const bool died = inRow && (p >= 0.0) && (p < 0x1p-800) && tame && (lambda <= 0.998f * rateF[n]);
                    if (died) p = 0.0; else laneBroken = inRow;
                }
                const unsigned brk = __ballot_sync(0xffffffffu, laneBroken);
                const int firstBrk = brk ? (__ffs(brk) - 1) : 32;
                broken = broken || lane >= firstBrk;
                const double pUse = (lane < firstBrk && inRow) ? p : 0.0;
                double Ssum = pUse, Us = (double)b * pUse;
#pragma unroll
                for (int o = 1; o < 32; o <<= 1) {
                    const double t1 = shfl_up_d(Ssum, o), t2 = shfl_up_d(Us, o);
                    if (lane >= o) { Ssum += t1; Us += t2; }
                }
                sum = carrySum + Ssum;
                uN = carryU + Us;
                carryP = __shfl_sync(0xffffffffu, p, 31);
                carrySum = __shfl_sync(0xffffffffu, sum, 31);
                carryU = __shfl_sync(0xffffffffu, uN, 31);
                if (brk) rowBroken = true;
                steps += 1;
            }
            // ---- candidate (r, b) ----------------------------------------------------------------------
            bool feasible = false; float itl = 0.0f, ttft = 0.0f, rho = 0.0f;
            int deferK = 0;
            if (inRow) {
                const float rateMax = rm.x;
                if (b > row.nGood) {                               // bad table entry: the literal path decides
                    const int k0 = atomicAdd(gp.slow_count, 1);
                    if (k0 < gp.slow_cap) gp.slow_list[k0] = (unsigned long long)(rowBase + n);
                }
                else if (!rateOk) scan_store_error(rc, n, WVA_CAND_ERR_RATE_LE0);
                else if (rc.rate > rateMax) scan_store_error(rc, n, WVA_CAND_ERR_RATE_MAX);
                else if (lambda < 0.0f) scan_store_error(rc, n, WVA_CAND_ERR_MODEL);
                else {
                    const int K = 11 * b;
                    SolveStats so;
                    bool certified = false;
                    if (!broken) {
                        if (stoppedLane) {
                            const double inServ = row.exInSys + oneMinusSumP * (double)b;
                            finish_stats(so, lambda, inServ, row.exInSys, 0.0f);
                            certified = true;
                        } else certified = cert_eval_fast(p, sum, uN, lam, rateD[n], rcp[n], b, K, lambda, so);
                    }
                    if (certified) {
                        okCount++;
                        algSteps += 2ULL * (unsigned long long)(K + 1);
                        feasible = scan_finish(pc, rc, so, n, (float)b, rateMax, rm.y, itl, ttft, rho);
                    } else deferK = K;                             // exact chain in the list kernels (appended below, warp-wide)
                }
            }
            // Uncertified candidates go to the exact-chain list as ONE block per warp and chunk, in lane order: such candidates
            // cluster (the aggregates of a row converge as b grows, so a limit on a float32 rounding boundary makes every large
            // b of that row ambiguous), and a list warp that gets 32 neighbours of one row runs them with one table, one
            // lambda and nearly equal trip counts.  Should the list ever be full (16 M entries) the literal-path list takes the
            // candidate (the host re-runs a slice whose literal list overflowed with a larger one).
            {
                const unsigned dm = __ballot_sync(0xffffffffu, deferK != 0);
                if (dm) {
                    const int leader = __ffs(dm) - 1;
                    int base = 0;
                    if (lane == leader) base = atomicAdd(gp.heavy_count, __popc(dm));
                    base = __shfl_sync(0xffffffffu, base, leader);
                    if (deferK) {
                        const int kk = base + __popc(dm & ((1u << lane) - 1u));
                        if (kk < gp.heavy_cap) { gp.heavy_list[kk] = (unsigned long long)(rowBase + n); gp.heavy_cost[kk] = (float)deferK; }
                        else { const int k2 = atomicAdd(gp.slow_count, 1); if (k2 < gp.slow_cap) gp.slow_list[k2] = (unsigned long long)(rowBase + n); }
                    }
                }
            }
            scan_row_best(best, rowHas, rc, feasible, n, itl, ttft, rho);
        }
    }
    scan_block_reduce(sys, gp, gs, k, slot, best.key, best.itl, best.ttft, best.rho, steps, algSteps, okCount, &sh_key, sh_cnt);
}

}  // namespace wva
