// tests/host_emul/emul_store.cpp — CPU build of the engine's integral store (semi-direct J/K, shell4.cuh: S4_STORE / S4_REPLAY).
//
// TEST TOOL, NOT A FALLBACK: the same engine body as the sm_100a kernels, run serially with the HostPolicy of emul.cpp.  Two Fock builds
// with two densities: the first runs the selected class jobs as a store pass, the second replays them; both are compared bitwise with
// direct builds by the tests.  The driver plays rank `rank` of `nranks` of a launch that deals FLAT units U = rank (mod nranks), job j's
// units starting at a flat offset unit0[j], exactly as k_shell4_multi does for the jobs of a group (k_shell4_one: offset 0).
#include "emul.cpp"

#include <cmath>

namespace {

constexpr int EMUL_CHUNK = 4;      // work items per unit

struct StoreSystem {
    PairTable PT;
    std::vector<double> boys, herm;
    ShellTab T;
    ShellSystem S;
};

struct StoreRun {                  // per job: mode, first double / first row of its share in the store, flat unit offset
    std::vector<int> mode;
    std::vector<long long> base, row0, unit0;
    int rank = 0, nranks = 1;
    double* store = nullptr;
    std::vector<int>* visits = nullptr;       // replay: digested rows
    std::vector<char>* stored = nullptr;      // store pass: rows written
    long long out_of_share = 0, only_store = 0;
};

// J/K (nD densities, output as emul_jk_shell4) of this rank's share of one build.  it_budget: chunk budget of the class tables (0 = default).
static void store_build(StoreSystem& Y, int ncart, int nD, const double* P, double tau, StoreRun& R, int it_budget, double* Jout, double* Kout) {
    ShellSystem& S = Y.S;
    const size_t nn = (size_t)ncart * ncart;
    std::vector<double> Pf(nD * nn), Psym(nD * nn);
    double dmax = 0.0;
    for (size_t x = 0; x < nD * nn; ++x) {
        const size_t i = (x % nn) / ncart, j = x % ncart;
        Pf[x] = S.fnorm[i] * S.fnorm[j] * P[x];
        dmax = std::max(dmax, std::fabs(P[x]));
    }
    for (int d = 0; d < nD; ++d)
        for (int i = 0; i < ncart; ++i)
            for (int j = 0; j < ncart; ++j) Psym[d * nn + (size_t)i * ncart + j] = Pf[d * nn + (size_t)i * ncart + j] + Pf[d * nn + (size_t)j * ncart + i];
    ShellData D;
    D.pairA = S.pairA.data(); D.pairB = S.pairB.data(); D.pair_rec = S.pair_rec.data(); D.rec = S.rec.data(); D.pairQ = S.pairQ.data();
    D.sh_ao = S.sh_ao.data(); D.boys = Y.boys.data(); D.herm = Y.herm.data();
    std::vector<long long> Jw(2 * nD * nn, 0), Kw(2 * nD * nn, 0);
    double* Jacc = reinterpret_cast<double*>(Jw.data()); double* Kacc = reinterpret_cast<double*>(Kw.data());
    D.fix_lo = (long long)(nD * nn);
    const char* enb = getenv("TUNA_EMUL_NB");
    const int NBATCH = enb ? atoi(enb) : 2;
    const int ncls = (int)S.classes.size();
    int job = 0;
    for (int cb = 0; cb < ncls; ++cb)
        for (int ck = 0; ck <= cb; ++ck, ++job) {
            Shell4Job J;
            J.La = S.classes[cb].La; J.Lb = S.classes[cb].Lb; J.Lc = S.classes[ck].La; J.Ld = S.classes[ck].Lb;
            J.nppAB = S.classes[cb].npp; J.nppCD = S.classes[ck].npp; J.chunk = EMUL_CHUNK; J.dbg_skip = 0; J.fill_scratch = nullptr; J.fill_base = 0; J.fill_pairs = nullptr;
            const char* ept = getenv("TUNA_EMUL_PSPLIT_TARGET");
            shell4_split(J, ept ? atoi(ept) : 16, true);
            J.bra_list = S.classes[cb].pairs.data(); J.ket_list = S.classes[ck].pairs.data();
            std::vector<long long> prefix;
            J.nitems = build_item_prefix(S, cb, ck, tau * 1e-3, prefix);
            J.item_prefix = prefix.data(); J.nbra = (int)S.classes[cb].pairs.size(); J.same_class = (cb == ck);
            Class4Host CH;
            if (it_budget > 0) build_class4_tables(Y.T, J.La, J.Lb, J.Lc, J.Ld, CH, it_budget, it_budget, 0);
            else build_class4_tables(Y.T, J.La, J.Lb, J.Lc, J.Ld, CH);
            J.ct = class4_view(CH, HostPtrOf());
            shell4_job_layout(J, nD);
            const int mode = R.mode[job];
            const long long nwi = J.nitems * J.psplit, nunits = (nwi + EMUL_CHUNK - 1) / EMUL_CHUNK;
            const StoreShare share = shell4_store_share(nwi, EMUL_CHUNK, R.unit0[job], R.rank, R.nranks);
            J.store = mode == S4_DIRECT ? nullptr : R.store;
            J.store_base = R.base[job]; J.store_mode = mode; J.store_nranks = R.nranks;
            J.store_unit0 = R.unit0[job]; J.store_ubase = share.ubase;
            std::vector<double> sm((size_t)4 * J.total);
            std::vector<unsigned> tab(CH.tab_words + 4);
            int tab_chunk = -1;
            for (long long u = 0; u < nunits; ++u) {
                if ((R.unit0[job] + u) % R.nranks != R.rank) continue;          // another rank's unit
                for (long long w0 = u * EMUL_CHUNK; w0 < std::min(nwi, (u + 1) * EMUL_CHUNK); w0 += NBATCH) {
                    Quartet4 hq[4];
                    for (int q = 0; q < 4; ++q) { hq[q] = Quartet4(); hq[q].active = 0; }
                    HostPolicy::row0() = w0;
                    const long long row = shell4_store_row<HostPolicy>(J, hq);
                    for (int q = 0; q < NBATCH && w0 + q < nwi; ++q) {
                        const long long wi = w0 + q, item = wi / J.psplit;
                        const int pchunk = (int)(wi - item * J.psplit);
                        int ib = 0, hi = J.nbra;
                        while (hi - ib > 1) { const int mid = (ib + hi) >> 1; if (prefix[mid] <= item) ib = mid; else hi = mid; }
                        const int AB = J.bra_list[ib], CD = J.ket_list[(int)(item - prefix[ib])];
                        Quartet4& h = hq[q];
                        // the device's per-build density test (shell4_unit); a store pass evaluates and stores the screened items too
                        h.active = (tau > 0.0 && S.pairQ[AB] * S.pairQ[CD] * dmax < tau) ? 0 : 1;
                        if (!h.active && mode == S4_STORE) { h.active = S4_ONLY_STORE; ++R.only_store; }
                        if (!h.active) continue;
                        if (mode != S4_DIRECT) {
                            if (row + q < 0 || row + q >= share.rows) { ++R.out_of_share; h.active = 0; continue; }
                            if (mode == S4_STORE) (*R.stored)[R.row0[job] + row + q] = 1;
                            if (mode == S4_REPLAY && h.active == 1) ++(*R.visits)[R.row0[job] + row + q];
                        }
                        h.shA = S.pairA[AB]; h.shB = S.pairB[AB]; h.shC = S.pairA[CD]; h.shD = S.pairB[CD];
                        h.ia0 = (pchunk / J.ksplit) * J.clen | ((pchunk % J.ksplit) * J.klen) << 16;
                        h.w = (h.shA == h.shB ? 0.5 : 1.0) * (h.shC == h.shD ? 0.5 : 1.0) * (AB == CD ? 0.5 : 1.0);
                        h.recA = S.pair_rec[AB]; h.recC = S.pair_rec[CD];
                        h.pA = S.rec[h.recA]; h.zA = S.rec[h.recA + 1]; h.pC = S.rec[h.recC]; h.zC = S.rec[h.recC + 1];
                    }
                    if (NBATCH == 4) shell4_quartets<HostPolicy, 4, true>(J, D, hq, sm.data(), tab.data(), tab_chunk, nD, Pf.data(), Psym.data(), Jacc, Kacc, ncart);
                    else if (NBATCH == 2) shell4_quartets<HostPolicy, 2, true>(J, D, hq, sm.data(), tab.data(), tab_chunk, nD, Pf.data(), Psym.data(), Jacc, Kacc, ncart);
                    else shell4_quartets<HostPolicy, 1, true>(J, D, hq, sm.data(), tab.data(), tab_chunk, nD, Pf.data(), Psym.data(), Jacc, Kacc, ncart);
                }
            }
        }
    for (int d = 0; d < nD; ++d)
        for (int i = 0; i < ncart; ++i)
            for (int j = 0; j < ncart; ++j) {
                const size_t ij = d * nn + (size_t)i * ncart + j, ji = d * nn + (size_t)j * ncart + i;
                const double ff = S.fnorm[i] * S.fnorm[j];
                Jout[ij] = ff * (fixed_value(Jw[ij], Jw[nD * nn + ij]) + fixed_value(Jw[ji], Jw[nD * nn + ji]));
                Kout[ij] = ff * (fixed_value(Kw[ij], Kw[nD * nn + ij]) + fixed_value(Kw[ji], Kw[nD * nn + ji]));
            }
}

}  // namespace

// Two builds of rank `rank` of `nranks`: P1 (store pass for the selected jobs) then P2 (replay of them).  select: 0 = no job stored (both
// builds direct), 1 = every job, 2 = every other job (a partial store).  Job j's units start at flat unit unit_shift * (j + 1) (0: every job
// has its own launch).  TUNA_EMUL_IT_BUDGET / TUNA_EMUL_IT_BUDGET_REPLAY: chunk budgets of the two builds' class tables (different chunk
// splits between store pass and replay).  J, K: [2][nD][n][n], this rank's partial J/K.  Each stored job gets exactly the rows
// shell4_store_share allocates for the rank, with NaN guard rows between the jobs.
// stats: [0] rows written by the store pass, [1] of those left NaN, [2] rows the replay digested more than once, [3] written rows not
// digested exactly once by the replay (0 when the replay build screens nothing out), [4] items screened out of the store pass's digestion
// but stored, [5] rows digested by the replay, [6] rows outside the rank's share (either build), [7] guard values overwritten.
extern "C" int emul_jk_shell4_store(int ncart, const double* oz, const int* lmn, const int* nprim, const int64_t* off, const double* exps,
                                    const double* ceff, int nD, const double* P1, const double* P2, double tau, int select, int rank, int nranks,
                                    int unit_shift, double* Jout, double* Kout, long long* stats) {
    HostBasis B = make_basis(ncart, oz, lmn, nprim, off, exps, ceff);
    StoreSystem Y;
    build_pair_table(B, Y.PT);
    build_boys_table(Y.boys);
    build_hermite_poly_table(Y.herm);
    std::vector<double> aoQ(Y.PT.npair);
    for (int64_t a = 0; a < Y.PT.npair; ++a) {
        PairClass ca{Y.PT.cls[a] & 255, (Y.PT.cls[a] >> 8) & 255, Y.PT.cls[a] >> 16};
        aoQ[a] = std::sqrt(std::fabs(eri_ao_quartet(Y.PT.pp.data() + Y.PT.ppoff[a] * PP_DOUBLES, Y.PT.npp[a], Y.PT.pp.data() + Y.PT.ppoff[a] * PP_DOUBLES,
                                                    Y.PT.npp[a], ca, ca, Y.boys.data(), Y.herm.data())));
    }
    build_shell_tab(Y.T);
    if (!detect_shells(B, Y.T, Y.S)) return 1;
    build_shell_pairs(Y.S, Y.T, Y.PT, aoQ, ncart);
    const ShellSystem& S = Y.S;
    const char* eb = getenv("TUNA_EMUL_IT_BUDGET");
    const char* ebr = getenv("TUNA_EMUL_IT_BUDGET_REPLAY");
    // the rank's share of every selected job (rows of the class's canonical integral count, independent of the chunk split) + a guard row
    const int ncls = (int)S.classes.size();
    StoreRun R1, R2;
    std::vector<std::pair<long long, long long>> guards;      // (first double, count) of the guard rows
    long long total = 0, nrows = 0;
    int job = 0;
    for (int cb = 0; cb < ncls; ++cb)
        for (int ck = 0; ck <= cb; ++ck, ++job) {
            Shell4Job J;
            J.nppAB = S.classes[cb].npp; J.nppCD = S.classes[ck].npp;
            const char* ept = getenv("TUNA_EMUL_PSPLIT_TARGET");
            shell4_split(J, ept ? atoi(ept) : 16, true);
            std::vector<long long> prefix;
            const long long nwi = build_item_prefix(S, cb, ck, tau * 1e-3, prefix) * J.psplit;
            Class4Host CH;
            build_class4_tables(Y.T, S.classes[cb].La, S.classes[cb].Lb, S.classes[ck].La, S.classes[ck].Lb, CH);
            const long long unit0 = (long long)unit_shift * (job + 1);
            const StoreShare share = shell4_store_share(nwi, EMUL_CHUNK, unit0, rank, nranks);
            const bool sel = select == 1 || (select == 2 && (job & 1) == 0);
            R1.mode.push_back(sel ? S4_STORE : S4_DIRECT);
            R2.mode.push_back(sel ? S4_REPLAY : S4_DIRECT);
            for (StoreRun* R : {&R1, &R2}) { R->base.push_back(total); R->row0.push_back(nrows); R->unit0.push_back(unit0); }
            if (sel) {
                total += share.rows * CH.nint; nrows += share.rows;
                guards.push_back({total, CH.nint});
                total += CH.nint;
            }
        }
    std::vector<double> store((size_t)std::max<long long>(total, 1), std::nan(""));
    std::vector<int> visits((size_t)std::max<long long>(nrows, 1), 0);
    std::vector<char> stored((size_t)std::max<long long>(nrows, 1), 0);
    const double guard = -12345.0;
    for (const auto& g : guards) for (long long e = 0; e < g.second; ++e) store[g.first + e] = guard;
    for (StoreRun* R : {&R1, &R2}) { R->rank = rank; R->nranks = nranks; R->store = store.data(); R->visits = &visits; R->stored = &stored; }
    const size_t nn = (size_t)ncart * ncart;
    store_build(Y, ncart, nD, P1, tau, R1, eb ? atoi(eb) : 0, Jout, Kout);
    long long written = 0, unwritten = 0;
    job = 0;
    for (int cb = 0; cb < ncls; ++cb)      // every row the store pass wrote must be complete
        for (int ck = 0; ck <= cb; ++ck, ++job) {
            if (R1.mode[job] != S4_STORE) continue;
            Class4Host CH;
            build_class4_tables(Y.T, S.classes[cb].La, S.classes[cb].Lb, S.classes[ck].La, S.classes[ck].Lb, CH);
            const long long end = (size_t)job + 1 < R1.row0.size() ? R1.row0[job + 1] : nrows;
            for (long long r = R1.row0[job]; r < end; ++r) {
                if (!stored[r]) continue;
                ++written;
                bool bad = false;
                for (int e = 0; e < CH.nint; ++e) bad |= std::isnan(store[R1.base[job] + (r - R1.row0[job]) * CH.nint + e]);
                unwritten += bad;
            }
        }
    store_build(Y, ncart, nD, P2, tau, R2, ebr ? atoi(ebr) : 0, Jout + nD * nn, Kout + nD * nn);
    long long twice = 0, not_once = 0, reads = 0, clobbered = 0;
    for (long long r = 0; r < nrows; ++r) {
        twice += visits[r] > 1; reads += visits[r];
        if (stored[r]) not_once += visits[r] != 1;
    }
    for (const auto& g : guards) for (long long e = 0; e < g.second; ++e) clobbered += store[g.first + e] != guard;
    if (stats) {
        stats[0] = written; stats[1] = unwritten; stats[2] = twice; stats[3] = not_once; stats[4] = R1.only_store; stats[5] = reads;
        stats[6] = R1.out_of_share + R2.out_of_share; stats[7] = clobbered;
    }
    return 0;
}
