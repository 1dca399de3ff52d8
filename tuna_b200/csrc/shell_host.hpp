// shell_host.hpp — host-side preparation for the shell-quartet engine (shell4.cuh): grouping the reference's
// per-component Basis list into shells, the primitive shell-pair records, pair classes and the job list.
// Built once per geometry.  Replaces, at shell granularity, the pair cache of
// TUNA/tuna_integrals/tuna_integral.pyx:1050-1128 and the pair12 >= pair34 double loop of :1312-1331.
#pragma once
#include <algorithm>
#include <cmath>
#include <cstdint>
#include <map>
#include <tuple>
#include <vector>

#include "pairtable.hpp"
#include "shell_jk.cuh"

namespace tuna {

struct HostShell {
    int L = 0, nprim = 0;
    double z = 0.0;
    std::vector<double> exps, coef;     // shell-level coefficients: ceff / f(component)
    int ao[SH_NCMAX];
    int filled = 0;
};

struct ShellSystem {
    bool ok = false;
    std::vector<HostShell> shells;
    std::vector<double> fnorm;           // per AO: f = 1 / sqrt((2l-1)!! (2m-1)!! (2n-1)!!)
    std::vector<int> sh_ao;              // [shell * SH_NCMAX + c]
    // shell pairs
    std::vector<int> pairA, pairB;
    std::vector<long long> pair_rec;
    std::vector<double> rec;
    std::vector<double> pairQ;
    // classes: key (La, Lb, npp)
    struct PairClassInfo { int La, Lb, npp; std::vector<int> pairs; };
    std::vector<PairClassInfo> classes;
};

inline double dfact_odd(int n) { double r = 1.0; while (n > 1) { r *= n; n -= 2; } return r; }

// Group the per-component list into full Cartesian shells.  Components of one shell need not be contiguous
// (DECONTRACT emits component-major order, tuna_molecule.py:557-565).  Returns false if the list is not a union of
// complete shells with a common radial part; the caller then uses the per-component kernels.
inline bool detect_shells(const HostBasis& B, const ShellTab& T, ShellSystem& S) {
    S = ShellSystem();
    const int n = B.ncart;
    S.fnorm.resize(n);
    std::map<std::tuple<int, int, int>, int> comp_index[SH_LMAX + 1];
    for (int L = 0; L <= SH_LMAX; ++L)
        for (int c = 0; c < T.nc[L]; ++c) comp_index[L][{T.lx[L][c], T.ly[L][c], T.lz[L][c]}] = c;
    std::map<std::tuple<double, int, int>, std::vector<int>> buckets;     // (z, L, nprim) -> candidate shells
    for (int i = 0; i < n; ++i) {
        const int l = B.lmn[3 * i], m = B.lmn[3 * i + 1], nn = B.lmn[3 * i + 2], L = l + m + nn;
        const double f = 1.0 / std::sqrt(dfact_odd(2 * l - 1) * dfact_odd(2 * m - 1) * dfact_odd(2 * nn - 1));
        S.fnorm[i] = f;
        const int c = comp_index[L][{l, m, nn}];
        const int np = B.nprim[i];
        auto& cand = buckets[{B.oz[i], L, np}];
        int found = -1;
        for (int s : cand) {
            HostShell& sh = S.shells[s];
            if (sh.ao[c] >= 0) continue;
            bool same = true;
            for (int k = 0; k < np && same; ++k) {
                const double ck = B.ceff[B.off[i] + k] / f;
                same = sh.exps[k] == B.exps[B.off[i] + k] && std::fabs(ck - sh.coef[k]) <= 1e-11 * std::fabs(sh.coef[k]);
            }
            if (same) { found = s; break; }
        }
        if (found < 0) {
            HostShell sh;
            sh.L = L; sh.nprim = np; sh.z = B.oz[i];
            for (int k = 0; k < np; ++k) { sh.exps.push_back(B.exps[B.off[i] + k]); sh.coef.push_back(B.ceff[B.off[i] + k] / f); }
            for (int k = 0; k < SH_NCMAX; ++k) sh.ao[k] = -1;
            found = (int)S.shells.size();
            S.shells.push_back(sh);
            cand.push_back(found);
        }
        S.shells[found].ao[c] = i;
        S.shells[found].filled++;
    }
    for (const HostShell& sh : S.shells)
        if (sh.filled != T.nc[sh.L]) return false;
    S.sh_ao.assign(S.shells.size() * SH_NCMAX, 0);
    for (size_t s = 0; s < S.shells.size(); ++s)
        for (int c = 0; c < T.nc[S.shells[s].L]; ++c) S.sh_ao[s * SH_NCMAX + c] = S.shells[s].ao[c];
    S.ok = true;
    return true;
}

// AO-level Schwarz factors (from the per-component pair table, already on the host) -> shell pairs, records, classes.
inline void build_shell_pairs(ShellSystem& S, const ShellTab& T, const PairTable& PT, const std::vector<double>& aoQ, int ncart) {
    const int ns = (int)S.shells.size();
    std::vector<int> lookup((size_t)ncart * ncart, -1);
    for (int64_t a = 0; a < PT.npair; ++a) {
        lookup[(size_t)PT.pi[a] * ncart + PT.pj[a]] = (int)a;
        lookup[(size_t)PT.pj[a] * ncart + PT.pi[a]] = (int)a;
    }
    S.pairA.clear(); S.pairB.clear(); S.pair_rec.clear(); S.pairQ.clear(); S.classes.clear();
    std::map<std::tuple<int, int, int>, int> class_of;
    long long rec_total = 0;
    for (int a = 0; a < ns; ++a)
        for (int b = 0; b <= a; ++b) {
            int A = a, Bs = b;
            if (S.shells[A].L < S.shells[Bs].L) std::swap(A, Bs);
            const HostShell& sa = S.shells[A];
            const HostShell& sb = S.shells[Bs];
            const int npp = sa.nprim * sb.nprim;
            double q = 0.0;
            for (int ca = 0; ca < T.nc[sa.L]; ++ca)
                for (int cb = 0; cb < T.nc[sb.L]; ++cb) q = std::max(q, aoQ[lookup[(size_t)sa.ao[ca] * ncart + sb.ao[cb]]]);
            const int id = (int)S.pairA.size();
            S.pairA.push_back(A); S.pairB.push_back(Bs); S.pairQ.push_back(q);
            S.pair_rec.push_back(rec_total);
            rec_total += (long long)npp * sp_rec_size(sa.L, sb.L);
            auto key = std::make_tuple(sa.L, sb.L, npp);
            auto it = class_of.find(key);
            if (it == class_of.end()) {
                it = class_of.emplace(key, (int)S.classes.size()).first;
                S.classes.push_back({sa.L, sb.L, npp, {}});
            }
            S.classes[it->second].pairs.push_back(id);
        }
    // deterministic class order: light to heavy; Schwarz-descending inside a class
    std::sort(S.classes.begin(), S.classes.end(), [](const ShellSystem::PairClassInfo& x, const ShellSystem::PairClassInfo& y) {
        return std::make_tuple(x.La + x.Lb, x.La, x.npp) < std::make_tuple(y.La + y.Lb, y.La, y.npp);
    });
    for (auto& c : S.classes)
        std::stable_sort(c.pairs.begin(), c.pairs.end(), [&](int x, int y) { return S.pairQ[x] > S.pairQ[y]; });
    S.rec.assign((size_t)rec_total, 0.0);
    const int np = (int)S.pairA.size();
    std::vector<std::vector<double>> scratch_of((size_t)host_threads());      // allocated outside the parallel region (see build_pair_table)
    for (auto& v : scratch_of) v.reserve(HERMITE_SCRATCH_DOUBLES);
#pragma omp parallel
    {
        std::vector<double>& scratch = scratch_of[(size_t)host_thread_id()];
#pragma omp for schedule(dynamic, 64)
        for (int id = 0; id < np; ++id) {
            const HostShell& sa = S.shells[S.pairA[id]];
            const HostShell& sb = S.shells[S.pairB[id]];
            const int La = sa.L, Lb = sb.L, Lab = La + Lb, rsz = sp_rec_size(La, Lb), nez = sp_ez_size(La, Lb), NT = Lab / 2 + 1;
            double* r = S.rec.data() + S.pair_rec[id];
            for (int ka = 0; ka < sa.nprim; ++ka)
                for (int kb = 0; kb < sb.nprim; ++kb, r += rsz) {
                    const double a = sa.exps[ka], b = sb.exps[kb], p = a + b;
                    r[0] = p; r[1] = (a * sa.z + b * sb.z) / p; r[2] = sa.coef[ka] * sb.coef[kb]; r[3] = 0.0;
                    hermite_table(La, Lb, sa.z - sb.z, a, b, scratch);
                    for (int i = 0; i <= La; ++i)
                        for (int j = 0; j <= Lb; ++j)
                            for (int t = 0; t <= i + j; ++t)
                                r[SP_HDR + (i * (Lb + 1) + j) * (Lab + 1) + t] = scratch[((size_t)i * (Lb + 1) + j) * (Lab + 2) + t];
                    hermite_table(Lab, 0, 0.0, a, b, scratch);
                    for (int nn = 0; nn <= Lab; ++nn)
                        for (int t = nn & 1; t <= nn; t += 2) r[SP_HDR + nez + nn * NT + (t >> 1)] = scratch[(size_t)nn * (Lab + 2) + t];
                }
        }
    }
}

// Kets kept per bra for one (bra class, ket class) job: Schwarz cut on the descending ket list; same class -> ket_pos <= bra_pos.
inline long long build_item_prefix(const ShellSystem& S, int cb, int ck, double tau_static, std::vector<long long>& prefix) {
    const auto& bra = S.classes[cb].pairs;
    const auto& ket = S.classes[ck].pairs;
    prefix.assign(bra.size() + 1, 0);
    for (size_t i = 0; i < bra.size(); ++i) {
        const double qb = S.pairQ[bra[i]];
        size_t lo = 0, hi = ket.size();       // first ket with Q_k * qb < tau_static
        if (tau_static > 0.0)
            while (lo < hi) {
                const size_t mid = (lo + hi) / 2;
                if (S.pairQ[ket[mid]] * qb >= tau_static) lo = mid + 1; else hi = mid;
            }
        else
            lo = ket.size();
        size_t keep = lo;
        if (cb == ck) keep = std::min(keep, i + 1);
        prefix[i + 1] = prefix[i] + (long long)keep;
    }
    return prefix.back();
}

// Cartesian->spherical rotation U (nbf x ncart, row-major) sliced by the engine's shells: block s holds the rows of the spherical
// functions built from shell s (columns = the shell's components in ShellTab order).  The spherical fill (shell4_fill_sph) rotates
// every shell quartet with these blocks, which is exact only when U is block-diagonal over the shells.
struct SphShells {
    std::vector<int> nsph;             // per shell: spherical functions (rows of its block)
    std::vector<int> sph;              // [shell * SH_NCMAX + k] -> spherical function index
    std::vector<int> uoff;             // per shell: first element of its block in u
    std::vector<double> u;             // blocks, each nsph x nc[L] row-major
    std::vector<int> par;              // per spherical function: x/y parity code (ShellTab::pg of every component in its row)
};

// True when every nonzero U[p][a] has p and a in the same shell, every row has a nonzero, all nonzeros of a row have one x/y parity
// (so parity-forbidden spherical elements are exact zeros), and no shell has more rows than components.  Fills Y when true.
inline bool build_sph_shells(const ShellSystem& S, const ShellTab& T, int nbf, int ncart, const double* U, SphShells& Y) {
    Y = SphShells();
    if (!S.ok) return false;
    const int ns = (int)S.shells.size();
    std::vector<int> shell_of(ncart, -1), comp_of(ncart, -1);
    for (int s = 0; s < ns; ++s)
        for (int c = 0; c < T.nc[S.shells[s].L]; ++c) { shell_of[S.shells[s].ao[c]] = s; comp_of[S.shells[s].ao[c]] = c; }
    Y.nsph.assign(ns, 0);
    Y.sph.assign((size_t)ns * SH_NCMAX, 0);
    Y.par.assign(nbf, 0);
    for (int p = 0; p < nbf; ++p) {
        int sh = -1, pg = -1;
        for (int a = 0; a < ncart; ++a) {
            if (U[(size_t)p * ncart + a] == 0.0) continue;
            const int g = T.pg[S.shells[shell_of[a]].L][comp_of[a]];
            if (sh < 0) { sh = shell_of[a]; pg = g; }
            if (shell_of[a] != sh || g != pg) return false;
        }
        if (sh < 0 || Y.nsph[sh] == T.nc[S.shells[sh].L]) return false;
        Y.sph[(size_t)sh * SH_NCMAX + Y.nsph[sh]++] = p;
        Y.par[p] = pg;
    }
    Y.uoff.assign(ns, 0);
    size_t total = 0;
    for (int s = 0; s < ns; ++s) { Y.uoff[s] = (int)total; total += (size_t)Y.nsph[s] * T.nc[S.shells[s].L]; }
    Y.u.assign(total, 0.0);
    for (int s = 0; s < ns; ++s) {
        const int nc = T.nc[S.shells[s].L];
        for (int k = 0; k < Y.nsph[s]; ++k)
            for (int c = 0; c < nc; ++c) Y.u[Y.uoff[s] + (size_t)k * nc + c] = U[(size_t)Y.sph[(size_t)s * SH_NCMAX + k] * ncart + S.shells[s].ao[c]];
    }
    return true;
}

struct HostPtrOf {
    template <class V> const typename V::value_type* operator()(const V& v) const { return v.data(); }
};

}  // namespace tuna
