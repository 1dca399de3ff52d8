// tests/host_emul/emul_sph.cpp — CPU build of the spherical fill (shell4_fill_sph of shell4.cuh, HostPolicy) on top of the fill-mode
// harness of emul.cpp, and of the block-diagonal check of U (build_sph_shells of shell_host.hpp).
//
// TEST TOOL, NOT A FALLBACK: the package never loads this library.
#include "emul.cpp"

static bool sph_setup(int ncart, const double* oz, const int* lmn, const int* nprim, const int64_t* off, const double* exps, const double* ceff,
                      HostBasis& B, ShellTab& T, ShellSystem& S) {
    B = make_basis(ncart, oz, lmn, nprim, off, exps, ceff);
    build_shell_tab(T);
    return detect_shells(B, T, S);
}

extern "C" int emul_sph_blocks_ok(int ncart, const double* oz, const int* lmn, const int* nprim, const int64_t* off, const double* exps,
                                  const double* ceff, int nbf, const double* U) {
    HostBasis B; ShellTab T; ShellSystem S; SphShells Y;
    if (!sph_setup(ncart, oz, lmn, nprim, off, exps, ceff, B, T, S)) return -1;
    return build_sph_shells(S, T, nbf, ncart, U, Y) ? 1 : 0;
}

// The spherical tensor (nbf^4) through the engine's fill mode and shell4_fill_sph.  `out` is not cleared: every element must be written.
extern "C" int emul_fill_sph(int ncart, const double* oz, const int* lmn, const int* nprim, const int64_t* off, const double* exps,
                             const double* ceff, int nbf, const double* U, double* out) {
    HostBasis B; ShellTab T; ShellSystem S; SphShells Ysh;
    if (!sph_setup(ncart, oz, lmn, nprim, off, exps, ceff, B, T, S)) return 1;
    if (!build_sph_shells(S, T, nbf, ncart, U, Ysh)) return 2;
    PairTable PT;
    build_pair_table(B, PT);
    std::vector<double> boys, herm;
    build_boys_table(boys);
    build_hermite_poly_table(herm);
    std::vector<double> aoQ(PT.npair, 1.0);
    build_shell_pairs(S, T, PT, aoQ, ncart);
    ShellData D;
    D.pairA = S.pairA.data(); D.pairB = S.pairB.data(); D.pair_rec = S.pair_rec.data(); D.rec = S.rec.data(); D.pairQ = S.pairQ.data();
    D.sh_ao = S.sh_ao.data(); D.boys = boys.data(); D.herm = herm.data(); D.fix_lo = 0;
    SphData Y;
    Y.nsph = Ysh.nsph.data(); Y.sph = Ysh.sph.data(); Y.uoff = Ysh.uoff.data(); Y.u = Ysh.u.data(); Y.par = Ysh.par.data();
    const int ncls = (int)S.classes.size();
    for (int cb = 0; cb < ncls; ++cb)
        for (int ck = 0; ck <= cb; ++ck) {
            Shell4Job J;
            J.La = S.classes[cb].La; J.Lb = S.classes[cb].Lb; J.Lc = S.classes[ck].La; J.Ld = S.classes[ck].Lb;
            J.nppAB = S.classes[cb].npp; J.nppCD = S.classes[ck].npp; J.chunk = 4; J.dbg_skip = 0;
            shell4_split(J, 16, true);
            J.bra_list = S.classes[cb].pairs.data(); J.ket_list = S.classes[ck].pairs.data();
            std::vector<long long> prefix;
            J.nitems = build_item_prefix(S, cb, ck, 0.0, prefix);
            J.item_prefix = prefix.data(); J.nbra = (int)S.classes[cb].pairs.size(); J.same_class = (cb == ck);
            Class4Host CH;
            build_class4_tables(T, J.La, J.Lb, J.Lc, J.Ld, CH, S4_IT_BUDGET, S4_S_BUDGET, 0, true);
            J.ct = class4_view(CH, HostPtrOf());
            shell4_job_layout(J, 0);
            std::vector<double> scratch((size_t)(J.nitems * J.psplit) * J.ct.nfill, -7.0);
            J.fill_scratch = scratch.data(); J.fill_base = 0;
            std::vector<int> fpairs;
            for (int ib = 0; ib < J.nbra; ++ib)
                for (long long k = 0; k < prefix[ib + 1] - prefix[ib]; ++k) { fpairs.push_back(J.bra_list[ib]); fpairs.push_back(J.ket_list[k]); }
            J.fill_pairs = fpairs.data();
            std::vector<double> sm((size_t)4 * J.total);
            std::vector<unsigned> tab(CH.tab_words + 4);
            int tab_chunk = -1;
            Quartet4 hq[4];
            const long long nwi = J.nitems * J.psplit;
            for (long long w0 = 0; w0 < nwi; w0 += 2) {
                for (int q = 0; q < 4; ++q) { hq[q] = Quartet4(); hq[q].active = 0; }
                for (int q = 0; q < 2 && w0 + q < nwi; ++q) {
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
                shell4_quartets<HostPolicy, 2>(J, D, hq, sm.data(), tab.data(), tab_chunk, 0, nullptr, nullptr, nullptr, nullptr, ncart);
            }
            const int nB = sph_ncart(J.Lb), ncd = sph_ncart(J.Lc) * sph_ncart(J.Ld);
            std::vector<double> cart((size_t)sph_ncart(J.La) * nB * ncd), X((size_t)nB * ncd), Yb((size_t)nB * ncd);
            for (long long item = 0; item < J.nitems; ++item)
                shell4_fill_sph<HostPolicy>(J, D, Y, item, S.fnorm.data(), cart.data(), X.data(), Yb.data(), out, nbf);
        }
    return 0;
}
