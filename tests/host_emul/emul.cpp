// tests/host_emul/emul.cpp — CPU unit-test harness for the kernel math of tuna_b200/csrc.
//
// TEST TOOL, NOT A FALLBACK: the development container has no GPU, so the `__host__ __device__` math in
// eri_core.cuh / pairtable.hpp is compiled here with g++ and checked against the oracle before GPU time
// is spent.  The package never loads this library; the product path is the CUDA library only.
#include <cstdint>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "../../tuna_b200/csrc/pairtable.hpp"

using namespace tuna;

static HostBasis make_basis(int ncart, const double* oz, const int* lmn, const int* nprim, const int64_t* off,
                            const double* exps, const double* ceff) {
    HostBasis B;
    B.ncart = ncart;
    B.oz.assign(oz, oz + ncart);
    B.lmn.assign(lmn, lmn + 3 * ncart);
    B.nprim.assign(nprim, nprim + ncart);
    B.off.assign(off, off + ncart);
    int64_t tot = 0;
    for (int i = 0; i < ncart; ++i) tot += nprim[i];
    B.exps.assign(exps, exps + tot);
    B.ceff.assign(ceff, ceff + tot);
    return B;
}

extern "C" {

double emul_boys(int M, int m, double T) {
    static std::vector<double> tab;
    if (tab.empty()) build_boys_table(tab);
    double F[BOYS_MMAX + 1];
    boys_fill(tab.data(), M, T, F);
    return F[m];
}

int emul_eri_fill(int ncart, const double* oz, const int* lmn, const int* nprim, const int64_t* off, const double* exps,
                  const double* ceff, double* out) {
    HostBasis B = make_basis(ncart, oz, lmn, nprim, off, exps, ceff);
    PairTable T;
    build_pair_table(B, T);
    std::vector<double> boys, herm;
    build_boys_table(boys);
    build_hermite_poly_table(herm);
    const int64_t n = ncart, n2 = n * n, n3 = n2 * n;
    std::memset(out, 0, sizeof(double) * n3 * n);
    for (int g = 0; g < 4; ++g) {
#pragma omp parallel for schedule(dynamic, 4)
        for (int64_t a = T.group_begin[g]; a < T.group_begin[g + 1]; ++a)
            for (int64_t b = T.group_begin[g]; b <= a; ++b) {
                PairClass ca{T.cls[a] & 255, (T.cls[a] >> 8) & 255, T.cls[a] >> 16};
                PairClass cb{T.cls[b] & 255, (T.cls[b] >> 8) & 255, T.cls[b] >> 16};
                double v = eri_ao_quartet(T.pp.data() + T.ppoff[a] * PP_DOUBLES, T.npp[a], T.pp.data() + T.ppoff[b] * PP_DOUBLES,
                                          T.npp[b], ca, cb, boys.data(), herm.data());
                int64_t i = T.pi[a], j = T.pj[a], k = T.pi[b], l = T.pj[b];
                out[i * n3 + j * n2 + k * n + l] = v; out[k * n3 + l * n2 + i * n + j] = v;
                out[j * n3 + i * n2 + l * n + k] = v; out[l * n3 + k * n2 + j * n + i] = v;
                out[j * n3 + i * n2 + k * n + l] = v; out[l * n3 + k * n2 + i * n + j] = v;
                out[i * n3 + j * n2 + l * n + k] = v; out[k * n3 + l * n2 + j * n + i] = v;
            }
    }
    return 0;
}
}

// ---- shell-quartet engine (shell_jk.cuh) with the serial HostPolicy ------------------------------------------------
#include "../../tuna_b200/csrc/density_split.hpp"
#include "../../tuna_b200/csrc/shell_host.hpp"
#include "../../tuna_b200/csrc/shell4_host.hpp"

struct HostPolicy {
    static constexpr int G = 1;
    static int lane() { return 0; }
    static void sync() {}
    static void sync_cta() {}
    static int cta_thread() { return 0; }
    static int cta_threads() { return 1; }
    static long long& row0() { static long long r = 0; return r; }           // fill mode: work item of the batch's first header (set by the driver)
    static long long work_item_of(const Shell4Job&, const Quartet4*) { return row0(); }
    static void accumulate(double* M, int idx, double v, long long fix_lo) {
        long long h, l;
        fixed_split(v, h, l);
        long long* W = reinterpret_cast<long long*>(M);
        W[idx] += h; W[fix_lo + idx] += l;
    }
};

// ---- generation-4 engine (shell4.cuh) with the serial HostPolicy: same driver, same conventions ---------------------------
extern "C" int emul_jk_shell4(int ncart, const double* oz, const int* lmn, const int* nprim, const int64_t* off, const double* exps,
                              const double* ceff, int nD, const double* P, double* Jout, double* Kout, double tau, long long* stats) {
    HostBasis B = make_basis(ncart, oz, lmn, nprim, off, exps, ceff);
    PairTable PT;
    build_pair_table(B, PT);
    std::vector<double> boys, herm;
    build_boys_table(boys);
    build_hermite_poly_table(herm);
    std::vector<double> aoQ(PT.npair);
    for (int64_t a = 0; a < PT.npair; ++a) {
        PairClass ca{PT.cls[a] & 255, (PT.cls[a] >> 8) & 255, PT.cls[a] >> 16};
        aoQ[a] = std::sqrt(std::fabs(eri_ao_quartet(PT.pp.data() + PT.ppoff[a] * PP_DOUBLES, PT.npp[a], PT.pp.data() + PT.ppoff[a] * PP_DOUBLES,
                                                    PT.npp[a], ca, ca, boys.data(), herm.data())));
    }
    ShellTab T;
    build_shell_tab(T);
    ShellSystem S;
    if (!detect_shells(B, T, S)) return 1;
    build_shell_pairs(S, T, PT, aoQ, ncart);
    const size_t nn = (size_t)ncart * ncart;
    std::vector<double> Pf(nD * nn), Jf(nD * nn, 0.0), Kf(nD * nn, 0.0);
    double dmax = 0.0;
    for (int d = 0; d < nD; ++d)
        for (int i = 0; i < ncart; ++i)
            for (int j = 0; j < ncart; ++j) {
                Pf[d * nn + (size_t)i * ncart + j] = S.fnorm[i] * S.fnorm[j] * P[d * nn + (size_t)i * ncart + j];
                dmax = std::max(dmax, std::fabs(P[d * nn + (size_t)i * ncart + j]));
            }
    double pmax, amax;      // the job lists are pre-screened with the bound the device build sets for this stack (plan_density)
    density_extrema(P, nD, ncart, &pmax, &amax);
    const double dens_bound = plan_density(nD, pmax, amax).dens_bound;
    std::vector<double> Psym(nD * nn);
    for (int d = 0; d < nD; ++d)
        for (int i = 0; i < ncart; ++i)
            for (int j = 0; j < ncart; ++j) Psym[d * nn + (size_t)i * ncart + j] = Pf[d * nn + (size_t)i * ncart + j] + Pf[d * nn + (size_t)j * ncart + i];
    ShellData D;
    D.pairA = S.pairA.data(); D.pairB = S.pairB.data(); D.pair_rec = S.pair_rec.data(); D.rec = S.rec.data(); D.pairQ = S.pairQ.data();
    D.sh_ao = S.sh_ao.data(); D.boys = boys.data(); D.herm = herm.data();
    // J/K accumulate as (high, low) 64-bit integer words (fixed_split), exactly as on the device
    std::vector<long long> Jw(2 * nD * nn, 0), Kw(2 * nD * nn, 0);
    double* Jacc = reinterpret_cast<double*>(Jw.data()); double* Kacc = reinterpret_cast<double*>(Kw.data());
    D.fix_lo = (long long)(nD * nn);
    long long nitems_total = 0, nskipped = 0, nint_total = 0, nterm_total = 0;
    const int ncls = (int)S.classes.size();
    for (int cb = 0; cb < ncls; ++cb)
        for (int ck = 0; ck <= cb; ++ck) {
            Shell4Job J;
            J.La = S.classes[cb].La; J.Lb = S.classes[cb].Lb; J.Lc = S.classes[ck].La; J.Ld = S.classes[ck].Lb;
            J.nppAB = S.classes[cb].npp; J.nppCD = S.classes[ck].npp; J.chunk = 4; J.dbg_skip = 0; J.fill_scratch = nullptr; J.fill_base = 0; J.fill_pairs = nullptr;
            {   // TUNA_EMUL_PSPLIT_TARGET: split contracted shell quartets into work items of primitive pairs, as the device launcher does
                const char* ept = getenv("TUNA_EMUL_PSPLIT_TARGET");
                const char* eks = getenv("TUNA_EMUL_KSPLIT");
                shell4_split(J, ept ? atoi(ept) : 16, !(eks && atoi(eks) == 0));
            }
            J.bra_list = S.classes[cb].pairs.data(); J.ket_list = S.classes[ck].pairs.data();
            std::vector<long long> prefix;
            J.nitems = build_item_prefix(S, cb, ck, tau / dens_bound, prefix);
            J.item_prefix = prefix.data(); J.nbra = (int)S.classes[cb].pairs.size(); J.same_class = (cb == ck);
            Class4Host CH;
            const char* eb = getenv("TUNA_EMUL_IT_BUDGET");      // small budgets force the multi-chunk path in tests
            const char* etm = getenv("TUNA_EMUL_TERM_MAX");       // 0 forces the separable digestion for every class
            const int tmax = etm ? atoi(etm) : S4_TERM_MAX;
            if (eb) build_class4_tables(T, J.La, J.Lb, J.Lc, J.Ld, CH, atoi(eb), atoi(eb), tmax); else build_class4_tables(T, J.La, J.Lb, J.Lc, J.Ld, CH, S4_IT_BUDGET, S4_S_BUDGET, tmax);
            J.ct = class4_view(CH, HostPtrOf());
            shell4_job_layout(J, nD);
            const char* enb = getenv("TUNA_EMUL_NB");
            const int NBATCH = enb ? atoi(enb) : 2;
            std::vector<double> sm((size_t)4 * J.total);
            std::vector<unsigned> tab(CH.tab_words + 4);
            int tab_chunk = -1;
            Quartet4 hq[4];
            for (int q = 0; q < 4; ++q) { hq[q] = Quartet4(); hq[q].active = 0; }
            int nb = 0;
            auto run_batch = [&]() {
                if (nb == 0) return;
                if (NBATCH == 4) shell4_quartets<HostPolicy, 4>(J, D, hq, sm.data(), tab.data(), tab_chunk, nD, Pf.data(), Psym.data(), Jacc, Kacc, ncart);
                else if (NBATCH == 2) shell4_quartets<HostPolicy, 2>(J, D, hq, sm.data(), tab.data(), tab_chunk, nD, Pf.data(), Psym.data(), Jacc, Kacc, ncart);
                else shell4_quartets<HostPolicy, 1>(J, D, hq, sm.data(), tab.data(), tab_chunk, nD, Pf.data(), Psym.data(), Jacc, Kacc, ncart);
                for (int q = 0; q < 4; ++q) hq[q].active = 0;
                nb = 0;
            };
            for (long long item = 0; item < J.nitems; ++item) {
                int ib = 0, hi = J.nbra;
                while (hi - ib > 1) { const int mid = (ib + hi) >> 1; if (prefix[mid] <= item) ib = mid; else hi = mid; }
                const int ik = (int)(item - prefix[ib]);
                const int AB = J.bra_list[ib], CD = J.ket_list[ik];
                if (tau > 0.0 && S.pairQ[AB] * S.pairQ[CD] * dmax < tau) { ++nskipped; continue; }
                double w = 1.0;
                if (S.pairA[AB] == S.pairB[AB]) w *= 0.5;
                if (S.pairA[CD] == S.pairB[CD]) w *= 0.5;
                if (AB == CD) w *= 0.5;
                for (int pchunk = 0; pchunk < J.psplit; ++pchunk) {
                    Quartet4 h;
                    h.active = 1; h.shA = S.pairA[AB]; h.shB = S.pairB[AB]; h.shC = S.pairA[CD]; h.shD = S.pairB[CD]; h.ia0 = (pchunk / J.ksplit) * J.clen | ((pchunk % J.ksplit) * J.klen) << 16; h.w = w;
                    h.recA = S.pair_rec[AB]; h.recC = S.pair_rec[CD];
                    h.pA = S.rec[h.recA]; h.zA = S.rec[h.recA + 1]; h.pC = S.rec[h.recC]; h.zC = S.rec[h.recC + 1];
                    hq[nb] = h;
                    if (++nb == NBATCH) run_batch();
                }
            }
            run_batch();
            nitems_total += J.nitems; nint_total += CH.nint; nterm_total += CH.nterms;
        }
    for (size_t x = 0; x < (size_t)nD * nn; ++x) { Jf[x] = fixed_value(Jw[x], Jw[nD * nn + x]); Kf[x] = fixed_value(Kw[x], Kw[nD * nn + x]); }
    for (int d = 0; d < nD; ++d)
        for (int i = 0; i < ncart; ++i)
            for (int j = 0; j < ncart; ++j) {
                const double ff = S.fnorm[i] * S.fnorm[j];
                Jout[d * nn + (size_t)i * ncart + j] = ff * (Jf[d * nn + (size_t)i * ncart + j] + Jf[d * nn + (size_t)j * ncart + i]);
                Kout[d * nn + (size_t)i * ncart + j] = ff * (Kf[d * nn + (size_t)i * ncart + j] + Kf[d * nn + (size_t)j * ncart + i]);
            }
    if (stats) { stats[0] = (long long)S.shells.size(); stats[1] = (long long)S.pairA.size(); stats[2] = nitems_total; stats[3] = nskipped; stats[4] = ncls; stats[5] = nint_total; stats[6] = nterm_total; }
    return 0;
}

// Work-item split of a contracted shell quartet (shell4_split): out = {psplit, clen, ksplit, klen}
extern "C" void emul_split(int nppAB, int nppCD, int target, int split_ket, int* out) {
    Shell4Job J;
    J.nppAB = nppAB; J.nppCD = nppCD;
    shell4_split(J, target, split_ket != 0);
    out[0] = J.psplit; out[1] = J.clen; out[2] = J.ksplit; out[3] = J.klen;
}

// Dense Cartesian ERI tensor through the engine's fill mode: every work item (shell quartet x primitive chunk) writes its integrals to
// a scratch row, shell4_fill_scatter sums the chunks and writes the eight images — the same two passes the device runs.
extern "C" int emul_fill_shell4(int ncart, const double* oz, const int* lmn, const int* nprim, const int64_t* off, const double* exps,
                                const double* ceff, double* out) {
    HostBasis B = make_basis(ncart, oz, lmn, nprim, off, exps, ceff);
    PairTable PT;
    build_pair_table(B, PT);
    std::vector<double> boys, herm;
    build_boys_table(boys);
    build_hermite_poly_table(herm);
    std::vector<double> aoQ(PT.npair, 1.0);             // no screening in fill mode; the factors only order the lists
    ShellTab T;
    build_shell_tab(T);
    ShellSystem S;
    if (!detect_shells(B, T, S)) return 1;
    build_shell_pairs(S, T, PT, aoQ, ncart);
    ShellData D;
    D.pairA = S.pairA.data(); D.pairB = S.pairB.data(); D.pair_rec = S.pair_rec.data(); D.rec = S.rec.data(); D.pairQ = S.pairQ.data();
    D.sh_ao = S.sh_ao.data(); D.boys = boys.data(); D.herm = herm.data(); D.fix_lo = 0;
    const long long n = ncart;
    std::memset(out, 0, sizeof(double) * n * n * n * n);      // parity-forbidden elements stay zero, as on the device
    const int ncls = (int)S.classes.size();
    for (int cb = 0; cb < ncls; ++cb)
        for (int ck = 0; ck <= cb; ++ck) {
            Shell4Job J;
            J.La = S.classes[cb].La; J.Lb = S.classes[cb].Lb; J.Lc = S.classes[ck].La; J.Ld = S.classes[ck].Lb;
            J.nppAB = S.classes[cb].npp; J.nppCD = S.classes[ck].npp; J.chunk = 4; J.dbg_skip = 0;
            {   // TUNA_EMUL_PSPLIT_TARGET: split contracted shell quartets into work items of primitive pairs, as the device launcher does
                const char* ept = getenv("TUNA_EMUL_PSPLIT_TARGET");
                const char* eks = getenv("TUNA_EMUL_KSPLIT");
                shell4_split(J, ept ? atoi(ept) : 16, !(eks && atoi(eks) == 0));
            }
            J.bra_list = S.classes[cb].pairs.data(); J.ket_list = S.classes[ck].pairs.data();
            std::vector<long long> prefix;
            J.nitems = build_item_prefix(S, cb, ck, 0.0, prefix);
            J.item_prefix = prefix.data(); J.nbra = (int)S.classes[cb].pairs.size(); J.same_class = (cb == ck);
            Class4Host CH;
            const char* eb = getenv("TUNA_EMUL_IT_BUDGET");
            if (eb) build_class4_tables(T, J.La, J.Lb, J.Lc, J.Ld, CH, atoi(eb), atoi(eb), 0, true);
            else build_class4_tables(T, J.La, J.Lb, J.Lc, J.Ld, CH, S4_IT_BUDGET, S4_S_BUDGET, 0, true);
            J.ct = class4_view(CH, HostPtrOf());
            shell4_job_layout(J, 0);
            std::vector<double> scratch((size_t)(J.nitems * J.psplit) * J.ct.nfill, -7.0);       // poisoned: every entry must be written
            J.fill_scratch = scratch.data(); J.fill_base = 0;
            std::vector<int> fpairs;
            for (int ib = 0; ib < J.nbra; ++ib)
                for (long long k = 0; k < prefix[ib + 1] - prefix[ib]; ++k) { fpairs.push_back(J.bra_list[ib]); fpairs.push_back(J.ket_list[k]); }
            J.fill_pairs = fpairs.data();
            const char* enb = getenv("TUNA_EMUL_NB");
            const int NBATCH = enb ? atoi(enb) : 2;
            std::vector<double> sm((size_t)4 * J.total);
            std::vector<unsigned> tab(CH.tab_words + 4);
            int tab_chunk = -1;
            Quartet4 hq[4];
            const long long nwi = J.nitems * J.psplit;
            for (long long w0 = 0; w0 < nwi; w0 += NBATCH) {
                for (int q = 0; q < 4; ++q) { hq[q] = Quartet4(); hq[q].active = 0; }
                for (int q = 0; q < NBATCH && w0 + q < nwi; ++q) {
                    const long long item = (w0 + q) / J.psplit;
                    const int pchunk = (int)((w0 + q) - item * J.psplit);
                    int ib = 0, hi = J.nbra;
                    while (hi - ib > 1) { const int mid = (ib + hi) >> 1; if (prefix[mid] <= item) ib = mid; else hi = mid; }
                    const int AB = J.bra_list[ib], CD = J.ket_list[(int)(item - prefix[ib])];
                    Quartet4& h = hq[q];
                    h.active = 1; h.shA = S.pairA[AB]; h.shB = S.pairB[AB]; h.shC = S.pairA[CD]; h.shD = S.pairB[CD]; h.ia0 = (pchunk / J.ksplit) * J.clen | ((pchunk % J.ksplit) * J.klen) << 16; h.w = 1.0;
                    h.recA = S.pair_rec[AB]; h.recC = S.pair_rec[CD];
                    h.pA = S.rec[h.recA]; h.zA = S.rec[h.recA + 1]; h.pC = S.rec[h.recC]; h.zC = S.rec[h.recC + 1];
                }
                HostPolicy::row0() = w0;
                if (NBATCH == 4) shell4_quartets<HostPolicy, 4>(J, D, hq, sm.data(), tab.data(), tab_chunk, 0, nullptr, nullptr, nullptr, nullptr, ncart);
                else if (NBATCH == 2) shell4_quartets<HostPolicy, 2>(J, D, hq, sm.data(), tab.data(), tab_chunk, 0, nullptr, nullptr, nullptr, nullptr, ncart);
                else shell4_quartets<HostPolicy, 1>(J, D, hq, sm.data(), tab.data(), tab_chunk, 0, nullptr, nullptr, nullptr, nullptr, ncart);
            }
            for (int mode = 0; mode < 4; ++mode)
                for (long long r = 0; r < J.nitems * J.ct.nfill; ++r) shell4_fill_scatter(J, D, r / J.ct.nfill, (int)(r % J.ct.nfill), mode, S.fnorm.data(), out, n);
        }
    return 0;
}

// ---- one-electron integrals (oneel_core.cuh), serial on the CPU ------------------------------------------------------
#include "../../tuna_b200/csrc/oneel_core.cuh"

extern "C" int emul_one_electron(int ncart, const double* oz, const int* lmn, const int* nprim, const int64_t* off, const double* exps,
                                 const double* ceff, int natoms, const double* atom_z, const double* atom_charge, const double* origin, double* S,
                                 double* T, double* V, double* D, double* Q) {
    std::vector<double> boys;
    build_boys_table(boys);
    const size_t n = (size_t)ncart, nn = n * n;
    for (int i = 0; i < ncart; ++i)
        for (int j = 0; j <= i; ++j) {
            const OneElPair o = one_electron_pair(lmn + 3 * i, oz[i], nprim[i], exps + off[i], ceff + off[i], lmn + 3 * j, oz[j], nprim[j], exps + off[j],
                                                  ceff + off[j], natoms, atom_z, atom_charge, origin, boys.data());
            const size_t ij = (size_t)i * n + j, ji = (size_t)j * n + i;
            S[ij] = S[ji] = o.s; T[ij] = T[ji] = o.t; V[ij] = V[ji] = o.v;
            for (int c = 0; c < 3; ++c) { D[c * nn + ij] = D[c * nn + ji] = o.d[c]; Q[c * nn + ij] = Q[c * nn + ji] = o.q[c]; }
        }
    return 0;
}

extern "C" int emul_cross_overlap(int n1, const double* oz1, const int* lmn1, const int* nprim1, const int64_t* off1, const double* exps1,
                                  const double* ceff1, int n2, const double* oz2, const int* lmn2, const int* nprim2, const int64_t* off2,
                                  const double* exps2, const double* ceff2, double* S12) {
    for (int i = 0; i < n1; ++i)
        for (int j = 0; j < n2; ++j)
            S12[(size_t)i * n2 + j] = overlap_pair(lmn1 + 3 * i, oz1[i], nprim1[i], exps1 + off1[i], ceff1 + off1[i], lmn2 + 3 * j, oz2[j], nprim2[j],
                                                   exps2 + off2[j], ceff2 + off2[j]);
    return 0;
}
