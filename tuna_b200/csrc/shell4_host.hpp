// shell4_host.hpp — per-class work tables of the generation-4 shell-quartet engine (shell4.cuh), built on the host once per
// angular class (La, Lb | Lc, Ld).  Everything that depends on Cartesian component indices only lives here, so the device code
// has no per-integral divisions or parity logic.  (Replaces, at shell granularity, the per-AO-pair caches of
// TUNA/tuna_integrals/tuna_integral.pyx:1050-1128 and the parity test of :1324-1327.)
#pragma once
#include <algorithm>
#include <map>
#include <tuple>
#include <vector>

#include "shell4.cuh"

namespace tuna {

struct Class4Host {
    int La, Lb, Lc, Ld;
    int nwork = 0, nstage = 0, nkst = 0, itmax = 0, zrow = 0, ssize = 0, nbeta = 0, ngamma = 0, nint = 0, ntab = 0;
    int jbrow_off = 0, jgcol_off = 0, jinfo_off = 0;
    unsigned char pgofs[4][8], gsz[4][4];
    int ncols[4], pgoff[4];
    Kind4 kind[4];
    std::vector<int> chunk_s0, chunk_t0, chunk_ni, chunk_row0;
    std::vector<unsigned> t_rt, t_xy, t_u, t_s, p4, tabs, acc, jst_ptr, jflush, terms, tptr;
    unsigned plan[64];
    int nterm2 = 0;                        // > 0: term mode (digestion lists in shared memory), pairs of terms
    int tab_words = 0;                     // words of the CTA's table area in either mode
    std::vector<unsigned short> pmap, omap, jst_list, wlist;
    std::vector<unsigned> wfl;
    std::vector<unsigned> fill;            // fill mode: {slot, a | b << 8 | c << 16 | d << 24} per parity-allowed component quartet, chunk by chunk
    std::vector<int> chunk_f0;
    std::vector<unsigned> fperm;           // [3][nfill] entry orders of the scatter modes 1..3 (c, b, a fastest)
    std::vector<unsigned> canon;           // integral store: canonical index of every integral slot, chunk by chunk (Class4Dev::canon)
    std::vector<int> chunk_c0;             //                 first canon entry of a chunk
    long long allowed = 0;                 // parity-allowed component quartets = integrals per shell quartet
    long long nterms = 0;                  // digestion terms (table statistics)
    bool terms_possible(int term_max) const { return nterms + nwork <= term_max && itmax < 65535 && nstage < 65535; }
    double uniq[6] = {0, 0, 0, 0, 0, 0};   // unique AO quartets a shell quartet stands for, by degeneracy case (as ClassTablesHost)
};

constexpr int S4_IT_BUDGET = 6144;     // doubles of shared memory for the integral buffer of a chunk
constexpr int S4_S_BUDGET = 4096;      // doubles for the S slice of a chunk
constexpr int S4_TERM_MAX = 4096;      // digestion terms up to which a single-chunk class keeps its term lists in shared memory (term mode)

inline void build_class4_tables(const ShellTab& T, int La, int Lb, int Lc, int Ld, Class4Host& C, int it_budget = S4_IT_BUDGET,
                                int s_budget = S4_S_BUDGET, int term_max = S4_TERM_MAX, bool with_fill = false) {
    C = Class4Host();
    C.La = La; C.Lb = Lb; C.Lc = Lc; C.Ld = Ld;
    const int Lsh[4] = {La, Lb, Lc, Ld};
    const int Lab = La + Lb, Lcd = Lc + Ld, Ltot = Lab + Lcd, NS = Ltot / 2 + 1, NGZ = (Lc + 1) * (Ld + 1);
    int nc[4];
    for (int s = 0; s < 4; ++s) nc[s] = T.nc[Lsh[s]];
    auto rc = [](int rsel, int r, int csel, int c) { return (unsigned short)((rsel << 5) | r | ((csel << 5 | c) << 8)); };

    // ---- components of every shell sorted by x/y parity group; groups padded to pairs --------------------------------------
    std::vector<int> sorted[4];      // padded-sorted position -> component, or -1 for a pad
    std::vector<int> pos_of[4];      // component -> padded-sorted position
    int padlen[4];
    for (int s = 0; s < 4; ++s) {
        pos_of[s].assign(nc[s], -1);
        for (int g = 0; g < 4; ++g) {
            C.pgofs[s][g] = (unsigned char)sorted[s].size();
            int cnt = 0;
            for (int c = 0; c < nc[s]; ++c)
                if (T.pg[Lsh[s]][c] == g) { pos_of[s][c] = (int)sorted[s].size(); sorted[s].push_back(c); ++cnt; }
            C.gsz[s][g] = (unsigned char)cnt;
            if (cnt & 1) sorted[s].push_back(-1);
        }
        C.pgofs[s][4] = (unsigned char)sorted[s].size();
        for (int g = 5; g < 8; ++g) C.pgofs[s][g] = C.pgofs[s][4];
        padlen[s] = (int)sorted[s].size();
    }

    // ---- pair functions ------------------------------------------------------------------------------------------------------
    // bra: beta = (sx12, sy12, az, bz); ket: gamma = (sx34, sy34, cz, dz); parity class pc = (sx & 1) * 2 + (sy & 1)
    struct PF { int sx, sy, z1, z2, pc; };
    std::map<std::tuple<int, int, int, int>, int> beta_of, gamma_of;
    std::vector<PF> betas, gammas;
    std::vector<int> bidx(nc[0] * nc[1]), gidx(nc[2] * nc[3]);
    for (int a = 0; a < nc[0]; ++a)
        for (int b = 0; b < nc[1]; ++b) {
            const int sx = T.lx[La][a] + T.lx[Lb][b], sy = T.ly[La][a] + T.ly[Lb][b];
            auto key = std::make_tuple(sx, sy, T.lz[La][a], T.lz[Lb][b]);
            auto it = beta_of.find(key);
            if (it == beta_of.end()) { it = beta_of.emplace(key, (int)betas.size()).first; betas.push_back({sx, sy, T.lz[La][a], T.lz[Lb][b], (sx & 1) * 2 + (sy & 1)}); }
            bidx[a * nc[1] + b] = it->second;
        }
    for (int c = 0; c < nc[2]; ++c)
        for (int d = 0; d < nc[3]; ++d) {
            const int sx = T.lx[Lc][c] + T.lx[Ld][d], sy = T.ly[Lc][c] + T.ly[Ld][d];
            auto key = std::make_tuple(sx, sy, T.lz[Lc][c], T.lz[Ld][d]);
            auto it = gamma_of.find(key);
            if (it == gamma_of.end()) { it = gamma_of.emplace(key, (int)gammas.size()).first; gammas.push_back({sx, sy, T.lz[Lc][c], T.lz[Ld][d], (sx & 1) * 2 + (sy & 1)}); }
            gidx[c * nc[3] + d] = it->second;
        }
    const int nbeta = (int)betas.size(), ngamma = (int)gammas.size();
    C.nbeta = nbeta; C.ngamma = ngamma;
    // column index of a gamma inside its parity class: ordered by (lz34, sx34, cz) so that the gz of one (lz34, sx34) are consecutive
    std::vector<int> Cg(ngamma, 0);
    for (int pc = 0; pc < 4; ++pc) {
        std::vector<int> ids;
        for (int g = 0; g < ngamma; ++g) if (gammas[g].pc == pc) ids.push_back(g);
        std::sort(ids.begin(), ids.end(), [&](int x, int y) {
            return std::make_tuple(gammas[x].z1 + gammas[x].z2, gammas[x].sx, gammas[x].z1) < std::make_tuple(gammas[y].z1 + gammas[y].z2, gammas[y].sx, gammas[y].z1);
        });
        for (size_t k = 0; k < ids.size(); ++k) Cg[ids[k]] = (int)k;
        C.ncols[pc] = (int)ids.size();
    }
    C.pgoff[0] = 0;
    for (int pc = 1; pc < 4; ++pc) C.pgoff[pc] = C.pgoff[pc - 1] + C.ncols[pc - 1];
    C.zrow = std::max(std::max(C.ncols[0], C.ncols[1]), std::max(C.ncols[2], C.ncols[3]));

    // ---- phase 1-2 work lists  ------------------------------------------------------------------------------
    for (int w = 0; w <= Ltot; ++w)
        for (int n = 0; 2 * n + w <= Ltot; ++n) C.t_rt.push_back((unsigned)(w * NS + n) | (unsigned)w << 16 | (unsigned)n << 24);
    for (int n12 = 0; n12 <= Lab; ++n12)
        for (int n34 = n12 & 1; n34 <= Lcd; n34 += 2)
            for (int m = n12 & 1; 2 * m <= n12 + n34; ++m)
                C.t_xy.push_back((unsigned)((n12 * (Lcd + 1) + n34) * NS + m) | (unsigned)n12 << 16 | (unsigned)n34 << 20 | (unsigned)m << 24);
    for (int v = 0; v <= Lab; ++v)
        for (int cz = 0; cz <= Lc; ++cz)
            for (int dz = 0; dz <= Ld; ++dz) {
                const int gz = cz * (Ld + 1) + dz, lz34 = cz + dz;
                for (int n = 0; 2 * n + v + lz34 <= Ltot; ++n) {
                    C.t_u.push_back((unsigned)((v * NGZ + gz) * NS + n) | (unsigned)(v * NS + n) << 16);
                    C.t_u.push_back((unsigned)(gz * (Lcd + 1)) | (unsigned)lz34 << 16);
                }
            }
    auto sort_pairs = [](std::vector<unsigned>& v, size_t lo, size_t hi, auto keyfn) {      // 2-word entries in [lo, hi), longest inner loop first
        std::vector<std::pair<unsigned, unsigned>> tmp;
        for (size_t i = lo; i < hi; i += 2) tmp.push_back({v[i], v[i + 1]});
        std::stable_sort(tmp.begin(), tmp.end(), [&](const auto& x, const auto& y) { return keyfn(x) > keyfn(y); });
        for (size_t i = 0; i < tmp.size(); ++i) { v[lo + 2 * i] = tmp[i].first; v[lo + 2 * i + 1] = tmp[i].second; }
    };
    std::stable_sort(C.t_rt.begin(), C.t_rt.end(), [](unsigned x, unsigned y) { return ((x >> 16) & 255) > ((y >> 16) & 255); });
    sort_pairs(C.t_u, 0, C.t_u.size(), [](const std::pair<unsigned, unsigned>& e) { return e.second >> 16; });

    // ---- chunks: runs of bra z rows (az, bz) whose integral slots and S slice fit the budgets ------------------------------------
    struct Row { int az, bz; };
    std::vector<Row> rows;
    for (int az = 0; az <= La; ++az)
        for (int bz = 0; bz <= Lb; ++bz) rows.push_back({az, bz});
    const int nrows = (int)rows.size();
    auto nzg = [&](int lz34) { int n = 0; for (int cz = 0; cz <= Lc; ++cz) { const int dz = lz34 - cz; if (dz >= 0 && dz <= Ld) ++n; } return n; };
    auto row_slots = [&](const Row& r) {         // integral slots of the betas of this row
        int n = 0;
        for (int b = 0; b < nbeta; ++b) if (betas[b].z1 == r.az && betas[b].z2 == r.bz) n += C.ncols[betas[b].pc];
        return n;
    };
    auto row_s = [&](const Row& r) {             // S entries of this row: blocks (lz12, lz34) of even total parity
        int n = 0;
        const int lz12 = r.az + r.bz;
        for (int lz34 = 0; lz34 <= Lcd; ++lz34)
            if (((Ltot - lz12 - lz34) & 1) == 0) n += nzg(lz34) * ((Ltot - lz12 - lz34) / 2 + 1);
        return n;
    };
    const int s_cap = std::min(s_budget, 65000);
    C.chunk_row0.push_back(0);
    {
        int cur_i = 0, cur_s = 0;
        for (int r = 0; r < nrows; ++r) {
            const int ni = row_slots(rows[r]), ns = row_s(rows[r]);
            if (r > C.chunk_row0.back() && (cur_i + ni > it_budget || cur_s + ns > s_cap)) { C.chunk_row0.push_back(r); cur_i = 0; cur_s = 0; }
            cur_i += ni; cur_s += ns;
        }
        C.chunk_row0.push_back(nrows);
    }
    const int nchunk = (int)C.chunk_row0.size() - 1;

    // ---- table area layout (words): T_AB[a][b''] T_BA[b][a''] T_CD[c][d''] T_DC[d][c''] JbRow JgCol jinfo -------------------------
    int toff[4];
    {
        int o = 0;
        toff[0] = o; o += nc[0] * padlen[1];
        toff[1] = o; o += nc[1] * padlen[0];
        toff[2] = o; o += nc[2] * padlen[3];
        toff[3] = o; o += nc[3] * padlen[2];
        C.jbrow_off = o; o += nbeta;
        C.jgcol_off = o; o += ngamma;
        C.jinfo_off = o; o += 16;
        C.ntab = (o + 1) & ~1;
    }
    C.tabs.assign((size_t)nchunk * C.ntab, 0u);
    // K blocks: kind k sums over (s, t): KAC (b, d), KAD (b, c), KBC (a, d), KBD (a, c); staged density P[t][s]
    const int ksel[4][4] = {{0, 2, 1, 3}, {0, 3, 1, 2}, {1, 2, 0, 3}, {1, 3, 0, 2}};      // {u, v, s, t} as shell selectors
    {
        int pb = 0;
        for (int k = 0; k < 4; ++k) {
            Kind4& K = C.kind[k];
            const int u = ksel[k][0], v = ksel[k][1], s = ksel[k][2], t = ksel[k][3];
            K.bra_tab = toff[u == 0 ? 0 : 1]; K.bra_pitch = padlen[s];
            K.ket_tab = toff[v == 2 ? 2 : 3]; K.ket_pitch = padlen[t];
            K.inner_ket = nc[t] >= nc[s] ? 1 : 0;
            K.oshell = K.inner_ket ? s : t; K.ishell = K.inner_ket ? t : s;
            K.pad_inner = padlen[K.ishell];
            K.pbase = pb;
            pb += padlen[K.oshell] * padlen[K.ishell];
        }
        C.nkst = pb;
    }
    for (int k = 0; k < 4; ++k)
        for (int g = 0; g < 4; ++g)
            for (int og = 0; og < 4; ++og) {
                const int os = C.kind[k].oshell, is = C.kind[k].ishell, ig = g ^ og;
                const int on = C.gsz[os][og], n2 = (C.pgofs[is][ig + 1] - C.pgofs[is][ig]) / 2;
                C.plan[(k * 4 + g) * 4 + og] = (on == 0 || n2 == 0) ? 0u : ((unsigned)C.pgofs[os][og] | (unsigned)on << 8 | (unsigned)C.pgofs[is][ig] << 16 | (unsigned)n2 << 24);
            }
    C.pmap.assign(C.nkst, 0xffff);
    for (int k = 0; k < 4; ++k) {
        const Kind4& K = C.kind[k];
        const int s = ksel[k][2], t = ksel[k][3];
        for (int o = 0; o < padlen[K.oshell]; ++o)
            for (int i = 0; i < padlen[K.ishell]; ++i) {
                const int co = sorted[K.oshell][o], ci = sorted[K.ishell][i];
                if (co < 0 || ci < 0) continue;
                const int cs = K.inner_ket ? co : ci, ct = K.inner_ket ? ci : co;      // components of s (bra side) and t (ket side)
                C.pmap[K.pbase + o * K.pad_inner + i] = rc(t, ct, s, cs);               // P[t][s]
            }
    }

    // ---- per chunk: row order, slots, S layout, phase 3 / 4 lists, digestion tables ---------------------------------------------
    std::vector<int> beta_chunk(nbeta, -1), beta_pb(nbeta, -1);     // chunk of a beta, its position in the Pb staging order
    std::vector<int> Rb0;                                            // integral-buffer rows of chunk 0 (term mode needs a single chunk)
    std::vector<int> canon_row(nbeta, 0);                            // canonical first index of a beta's row: betas in class order
    for (int b = 1; b < nbeta; ++b) canon_row[b] = canon_row[b - 1] + C.ncols[betas[b - 1].pc];
    int pb_run = 0;
    C.chunk_s0.push_back(0); C.chunk_t0.push_back(0);
    for (int ch = 0; ch < nchunk; ++ch) {
        unsigned* tab = C.tabs.data() + (size_t)ch * C.ntab;
        const int r0 = C.chunk_row0[ch], r1 = C.chunk_row0[ch + 1];
        auto in_chunk = [&](const PF& b) {
            for (int r = r0; r < r1; ++r) if (rows[r].az == b.z1 && rows[r].bz == b.z2) return r - r0;
            return -1;
        };
        // rows of the integral buffer: the chunk's betas grouped by parity class
        std::vector<int> Rb(nbeta, -1);
        int slots = 0;
        for (int pc = 0; pc < 4; ++pc) {
            tab[C.jinfo_off + 4 * pc] = (unsigned)slots;
            tab[C.jinfo_off + 4 * pc + 2] = (unsigned)pb_run;
            int n = 0;
            for (int b = 0; b < nbeta; ++b) {
                if (betas[b].pc != pc || in_chunk(betas[b]) < 0) continue;
                Rb[b] = slots; slots += C.ncols[pc];
                beta_chunk[b] = ch; beta_pb[b] = pb_run++;
                ++n;
            }
            tab[C.jinfo_off + 4 * pc + 1] = (unsigned)n;
        }
        if (ch == 0) Rb0 = Rb;
        C.chunk_c0.push_back((int)C.canon.size());
        C.canon.resize(C.canon.size() + slots);
        for (int b = 0; b < nbeta; ++b)
            if (Rb[b] >= 0)
                for (int k = 0; k < C.ncols[betas[b].pc]; ++k) C.canon[C.chunk_c0.back() + Rb[b] + k] = (unsigned)(canon_row[b] + k);
        C.chunk_ni.push_back(slots);
        C.itmax = std::max(C.itmax, slots);
        C.nint += slots;
        // S slice: blocks (lz12, lz34) of even parity, layout [n][zc], zc = (row of the chunk with az + bz = lz12) x (gz with cz + dz = lz34)
        struct Block { int lz12, lz34, sbase, nzc, nn; std::vector<std::pair<int, int>> zc; };     // zc: (row index in chunk, gz)
        std::vector<Block> blocks;
        int srun = 0;
        for (int lz12 = 0; lz12 <= Lab; ++lz12)
            for (int lz34 = 0; lz34 <= Lcd; ++lz34) {
                if ((Ltot - lz12 - lz34) & 1) continue;
                Block B;
                B.lz12 = lz12; B.lz34 = lz34; B.nn = (Ltot - lz12 - lz34) / 2 + 1;
                for (int r = r0; r < r1; ++r) {
                    if (rows[r].az + rows[r].bz != lz12) continue;
                    for (int cz = 0; cz <= Lc; ++cz) { const int dz = lz34 - cz; if (dz >= 0 && dz <= Ld) B.zc.push_back({r - r0, cz * (Ld + 1) + dz}); }
                }
                if (B.zc.empty()) continue;
                B.nzc = (int)B.zc.size(); B.sbase = srun; srun += B.nzc * B.nn;
                blocks.push_back(B);
            }
        C.ssize = std::max(C.ssize, srun);
        // phase 3 entries
        for (const Block& B : blocks)
            for (int z = 0; z < B.nzc; ++z) {
                const Row& rw = rows[r0 + B.zc[z].first];
                const int gz = B.zc[z].second;
                for (int n = 0; n < B.nn; ++n) {
                    C.t_s.push_back((unsigned)(B.sbase + n * B.nzc + z) | (unsigned)(gz * NS + n) << 16);
                    C.t_s.push_back((unsigned)((rw.az * (Lb + 1) + rw.bz) * (Lab + 1)) | (unsigned)B.lz12 << 16);
                }
            }
        sort_pairs(C.t_s, 2 * (size_t)C.chunk_s0.back(), C.t_s.size(), [](const std::pair<unsigned, unsigned>& e) { return e.second >> 16; });
        C.chunk_s0.push_back((int)C.t_s.size() / 2);
        // phase 4 tiles
        struct Tile { unsigned w[4]; int ny, nx; };
        std::vector<Tile> tiles;
        for (const Block& B : blocks) {
            const int rx12 = Lab - B.lz12, rx34 = Lcd - B.lz34;
            for (int sx12 = 0; sx12 <= rx12; ++sx12)
                for (int sx34 = sx12 & 1; sx34 <= rx34; sx34 += 2) {
                    const int sy12 = rx12 - sx12, sy34 = rx34 - sx34;
                    const unsigned xoff = (sx12 * (Lcd + 1) + sx34) * NS, yoff = (sy12 * (Lcd + 1) + sy34) * NS;
                    const int mx0 = sx12 & 1, mx1 = (sx12 + sx34) >> 1, my0 = sy12 & 1, my1 = (sy12 + sy34) >> 1;
                    for (int z = 0; z < B.nzc; z += 2) {
                        const int cnt = std::min(2, B.nzc - z);
                        unsigned slot[2] = {0, 0};
                        for (int j = 0; j < cnt; ++j) {
                            const Row& rw = rows[r0 + B.zc[z + j].first];
                            const int gz = B.zc[z + j].second, cz = gz / (Ld + 1), dz = gz % (Ld + 1);
                            const int b = beta_of.at(std::make_tuple(sx12, sy12, rw.az, rw.bz)), g = gamma_of.at(std::make_tuple(sx34, sy34, cz, dz));
                            slot[j] = (unsigned)(Rb[b] + Cg[g]);
                        }
                        Tile t;
                        t.w[0] = xoff | yoff << 16;
                        t.w[1] = (unsigned)(B.sbase + z) | (unsigned)B.nzc << 16;
                        t.w[2] = (unsigned)mx0 | (unsigned)mx1 << 4 | (unsigned)my0 << 8 | (unsigned)(my1 - my0 + 1) << 12 | (unsigned)cnt << 16;
                        t.w[3] = slot[0] | slot[1] << 16;
                        t.ny = my1 - my0 + 1; t.nx = mx1 - mx0 + 1;
                        tiles.push_back(t);
                    }
                }
        }
        std::stable_sort(tiles.begin(), tiles.end(), [](const Tile& x, const Tile& y) { return x.ny * 16 + x.nx > y.ny * 16 + y.nx; });
        for (const Tile& t : tiles) for (int k = 0; k < 4; ++k) C.p4.push_back(t.w[k]);
        C.chunk_t0.push_back((int)C.p4.size() / 4);
        // digestion tables of the chunk
        for (int a = 0; a < nc[0]; ++a)
            for (int b = 0; b < nc[1]; ++b) {
                const int be = bidx[a * nc[1] + b];
                const unsigned v = Rb[be] >= 0 ? (unsigned)Rb[be] : S4_ABSENT;
                tab[toff[0] + a * padlen[1] + pos_of[1][b]] = v;
                tab[toff[1] + b * padlen[0] + pos_of[0][a]] = v;
            }
        for (int c = 0; c < nc[2]; ++c)
            for (int d = 0; d < nc[3]; ++d) {
                const unsigned v = (unsigned)Cg[gidx[c * nc[3] + d]];
                tab[toff[2] + c * padlen[3] + pos_of[3][d]] = v;
                tab[toff[3] + d * padlen[2] + pos_of[2][c]] = v;
            }
        for (int b = 0; b < nbeta; ++b) tab[C.jbrow_off + b] = Rb[b] >= 0 ? (unsigned)Rb[b] : S4_ABSENT;
        for (int g = 0; g < ngamma; ++g) tab[C.jgcol_off + g] = (unsigned)Cg[g];
        // fill list of the chunk: every allowed component quartet whose bra pair function lives in this chunk (d fastest)
        if (with_fill) {
            C.chunk_f0.push_back((int)C.fill.size() / 2);
            for (int a = 0; a < nc[0]; ++a) for (int b = 0; b < nc[1]; ++b) {
                const int be = bidx[a * nc[1] + b];
                if (Rb[be] < 0) continue;
                for (int c = 0; c < nc[2]; ++c) for (int d = 0; d < nc[3]; ++d) {
                    if ((T.pg[La][a] ^ T.pg[Lb][b] ^ T.pg[Lc][c] ^ T.pg[Ld][d]) != 0) continue;
                    C.fill.push_back((unsigned)(Rb[be] + Cg[gidx[c * nc[3] + d]]));
                    C.fill.push_back((unsigned)a | (unsigned)b << 8 | (unsigned)c << 16 | (unsigned)d << 24);
                }
            }
        }
    }
    C.chunk_c0.push_back((int)C.canon.size());
    if (with_fill) {
        C.chunk_f0.push_back((int)C.fill.size() / 2);
        const int nf = (int)C.fill.size() / 2;
        std::vector<unsigned> idx(nf);
        for (int mode = 1; mode <= 3; ++mode) {
            for (int e = 0; e < nf; ++e) idx[e] = (unsigned)e;
            auto key = [&](unsigned e) {
                const unsigned m = C.fill[2 * e + 1], a = m & 255, b = (m >> 8) & 255, c = (m >> 16) & 255, d = m >> 24;
                return mode == 1 ? std::make_tuple(a, b, d, c) : mode == 2 ? std::make_tuple(c, d, a, b) : std::make_tuple(c, d, b, a);
            };
            std::stable_sort(idx.begin(), idx.end(), [&](unsigned x, unsigned y) { return key(x) < key(y); });
            C.fperm.insert(C.fperm.end(), idx.begin(), idx.end());
        }
    }

    // ---- staging of the pair-function densities: Pg in (parity class, column) order, then Pb in the chunks' row order ----------------
    C.nstage = C.nkst + ngamma + nbeta;
    {
        std::vector<std::vector<unsigned short>> lists(ngamma + nbeta);
        for (int c = 0; c < nc[2]; ++c)
            for (int d = 0; d < nc[3]; ++d) { const int g = gidx[c * nc[3] + d]; lists[C.pgoff[gammas[g].pc] + Cg[g]].push_back(rc(2, c, 3, d)); }
        for (int a = 0; a < nc[0]; ++a)
            for (int b = 0; b < nc[1]; ++b) lists[ngamma + beta_pb[bidx[a * nc[1] + b]]].push_back(rc(0, a, 1, b));
        C.jst_ptr.push_back(0);
        for (auto& l : lists) { C.jst_list.insert(C.jst_list.end(), l.begin(), l.end()); C.jst_ptr.push_back((unsigned)C.jst_list.size()); }
    }

    // ---- work list: K accumulators of the four blocks, then the pair functions; heaviest first --------------------------------------
    struct Work { unsigned w0, w1; long long cost; unsigned short om; int jb, jg; };
    std::vector<Work> work;
    const int nK[4][2] = {{nc[0], nc[2]}, {nc[0], nc[3]}, {nc[1], nc[2]}, {nc[1], nc[3]}};
    for (int k = 0; k < 4; ++k) {
        const int us = ksel[k][0], vs = ksel[k][1], ss = ksel[k][2], ts = ksel[k][3];
        for (int u = 0; u < nK[k][0]; ++u)
            for (int v = 0; v < nK[k][1]; ++v) {
                const int g = T.pg[Lsh[us]][u] ^ T.pg[Lsh[vs]][v];
                long long cost = 0;
                for (int og = 0; og < 4; ++og) cost += (long long)C.gsz[ss][og] * C.gsz[ts][g ^ og];
                C.nterms += cost;
                work.push_back({(unsigned)k | (unsigned)g << 4 | (unsigned)u << 8 | (unsigned)v << 16, 0u, cost, rc(us, u, vs, v), -1, -1});
            }
    }
    for (int b = 0; b < nbeta; ++b) { work.push_back({4u | (unsigned)betas[b].pc << 4, (unsigned)b, (long long)C.ncols[betas[b].pc], 0xffff, b, -1}); C.nterms += C.ncols[betas[b].pc]; }
    {
        int nb_pc[4] = {0, 0, 0, 0};
        for (int b = 0; b < nbeta; ++b) ++nb_pc[betas[b].pc];
        for (int g = 0; g < ngamma; ++g) { work.push_back({5u | (unsigned)gammas[g].pc << 4, (unsigned)g, (long long)nb_pc[gammas[g].pc], 0xffff, -1, g}); C.nterms += nb_pc[gammas[g].pc]; }
    }
    // warps should be homogeneous: order by (kind, parity), heavier kinds first
    std::stable_sort(work.begin(), work.end(), [](const Work& x, const Work& y) {
        if (x.cost != y.cost) return x.cost > y.cost;
        return (x.w0 & 255u) < (y.w0 & 255u);
    });
    C.nwork = (int)work.size();
    std::vector<int> pos_jb(nbeta, 0), pos_jg(ngamma, 0);
    for (int w = 0; w < C.nwork; ++w) {
        C.acc.push_back(work[w].w0); C.acc.push_back(work[w].w1);
        C.omap.push_back(work[w].om);
        if (work[w].jb >= 0) pos_jb[work[w].jb] = w;
        if (work[w].jg >= 0) pos_jg[work[w].jg] = w;
    }
    for (int a = 0; a < nc[0]; ++a)
        for (int b = 0; b < nc[1]; ++b) C.jflush.push_back((unsigned)rc(0, a, 1, b) | (unsigned)pos_jb[bidx[a * nc[1] + b]] << 16);
    for (int c = 0; c < nc[2]; ++c)
        for (int d = 0; d < nc[3]; ++d) C.jflush.push_back((unsigned)rc(2, c, 3, d) | (unsigned)pos_jg[gidx[c * nc[3] + d]] << 16);

    // ---- term mode: light single-chunk classes digest through explicit (slot, density entry) lists held in shared memory --------------
    C.tab_words = C.ntab;
    if (nchunk == 1 && C.terms_possible(term_max)) {
        // compact staging: P[d][b], P[c][b], P[d][a], P[c][a] without padding, then Pg and Pb as above
        const int pbo[4] = {0, nc[3] * nc[1], nc[3] * nc[1] + nc[2] * nc[1], nc[3] * nc[1] + nc[2] * nc[1] + nc[3] * nc[0]};
        const int nk = pbo[3] + nc[2] * nc[0];
        C.pmap.assign(nk, 0);
        for (int d = 0; d < nc[3]; ++d) for (int b = 0; b < nc[1]; ++b) C.pmap[pbo[0] + d * nc[1] + b] = rc(3, d, 1, b);
        for (int c = 0; c < nc[2]; ++c) for (int b = 0; b < nc[1]; ++b) C.pmap[pbo[1] + c * nc[1] + b] = rc(2, c, 1, b);
        for (int d = 0; d < nc[3]; ++d) for (int a = 0; a < nc[0]; ++a) C.pmap[pbo[2] + d * nc[0] + a] = rc(3, d, 0, a);
        for (int c = 0; c < nc[2]; ++c) for (int a = 0; a < nc[0]; ++a) C.pmap[pbo[3] + c * nc[0] + a] = rc(2, c, 0, a);
        C.nkst = nk;
        C.nstage = nk + ngamma + nbeta;
        std::vector<std::vector<unsigned>> lists(C.nwork);
        auto slot_of = [&](int a, int b, int c, int d) { return (unsigned)(Rb0[bidx[a * nc[1] + b]] + Cg[gidx[c * nc[3] + d]]); };
        std::vector<int> pos_k[4];
        for (int k = 0; k < 4; ++k) pos_k[k].assign(nK[k][0] * nK[k][1], -1);
        for (int w = 0; w < C.nwork; ++w) {
            const unsigned w0 = work[w].w0;
            if ((w0 & 15u) < 4u) pos_k[w0 & 15u][((w0 >> 8) & 255u) * nK[w0 & 15u][1] + ((w0 >> 16) & 255u)] = w;
        }
        for (int a = 0; a < nc[0]; ++a) for (int b = 0; b < nc[1]; ++b) for (int c = 0; c < nc[2]; ++c) for (int d = 0; d < nc[3]; ++d) {
            if ((T.pg[La][a] ^ T.pg[Lb][b] ^ T.pg[Lc][c] ^ T.pg[Ld][d]) != 0) continue;
            const unsigned sl = slot_of(a, b, c, d);
            lists[pos_k[0][a * nc[2] + c]].push_back(sl | (unsigned)(pbo[0] + d * nc[1] + b) << 16);     // KAC += I P[d][b]
            lists[pos_k[1][a * nc[3] + d]].push_back(sl | (unsigned)(pbo[1] + c * nc[1] + b) << 16);     // KAD += I P[c][b]
            lists[pos_k[2][b * nc[2] + c]].push_back(sl | (unsigned)(pbo[2] + d * nc[0] + a) << 16);     // KBC += I P[d][a]
            lists[pos_k[3][b * nc[3] + d]].push_back(sl | (unsigned)(pbo[3] + c * nc[0] + a) << 16);     // KBD += I P[c][a]
        }
        for (int b = 0; b < nbeta; ++b)
            for (int g = 0; g < ngamma; ++g) {
                if (betas[b].pc != gammas[g].pc) continue;
                const unsigned sl = (unsigned)(Rb0[b] + Cg[g]);
                lists[pos_jb[b]].push_back(sl | (unsigned)(nk + C.pgoff[gammas[g].pc] + Cg[g]) << 16);     // Jb[beta]  += I Pg[gamma]
                lists[pos_jg[g]].push_back(sl | (unsigned)(nk + ngamma + beta_pb[b]) << 16);               // Jg[gamma] += I Pb[beta]
            }
        for (int w = 0; w < C.nwork; ++w) {
            if (lists[w].size() & 1) lists[w].push_back((unsigned)C.itmax);                                // pad: zero row, density entry 0
            C.tptr.push_back((unsigned)(C.terms.size() / 2) | (unsigned)(lists[w].size() / 2) << 20);
            C.terms.insert(C.terms.end(), lists[w].begin(), lists[w].end());
        }
        C.nterm2 = (int)C.terms.size() / 2;
        // flush lists: one target per K accumulator, the component pairs of the pair function for a J accumulator
        std::vector<std::vector<unsigned short>> fls(C.nwork);
        for (int w = 0; w < C.nwork; ++w) if (C.omap[w] != 0xffff) fls[w].push_back(C.omap[w]);
        for (int a = 0; a < nc[0]; ++a) for (int b = 0; b < nc[1]; ++b) fls[pos_jb[bidx[a * nc[1] + b]]].push_back(rc(0, a, 1, b));
        for (int c = 0; c < nc[2]; ++c) for (int d = 0; d < nc[3]; ++d) fls[pos_jg[gidx[c * nc[3] + d]]].push_back(rc(2, c, 3, d));
        for (int w = 0; w < C.nwork; ++w) {
            C.wfl.push_back((unsigned)C.wlist.size() | (unsigned)fls[w].size() << 16 | (C.omap[w] == 0xffff ? 1u << 31 : 0u));
            C.wlist.insert(C.wlist.end(), fls[w].begin(), fls[w].end());
        }
        C.tab_words = 4 * C.nterm2 + 2 * C.nwork + ((int)C.wlist.size() + 1) / 2;
    }

    // ---- statistics ------------------------------------------------------------------------------------------------------------
    for (int a = 0; a < nc[0]; ++a) for (int b = 0; b < nc[1]; ++b) for (int c = 0; c < nc[2]; ++c) for (int d = 0; d < nc[3]; ++d)
        if ((T.pg[La][a] ^ T.pg[Lb][b] ^ T.pg[Lc][c] ^ T.pg[Ld][d]) == 0) ++C.allowed;
    auto count = [&](bool ab, bool cd, bool diag) {
        double n = 0;
        for (int a = 0; a < nc[0]; ++a) for (int b = 0; b < nc[1]; ++b) {
            if (ab && b > a) continue;
            for (int c = 0; c < nc[2]; ++c) for (int d = 0; d < nc[3]; ++d) {
                if (cd && d > c) continue;
                if ((T.pg[La][a] ^ T.pg[Lb][b] ^ T.pg[Lc][c] ^ T.pg[Ld][d]) != 0) continue;
                if (diag && (c * nc[3] + d) > (a * nc[1] + b)) continue;
                n += 1;
            }
        }
        return n;
    };
    C.uniq[0] = count(false, false, false); C.uniq[1] = count(true, false, false); C.uniq[2] = count(false, true, false);
    C.uniq[3] = count(true, true, false);
    C.uniq[4] = (La == Lc && Lb == Ld) ? count(false, false, true) : 0;
    C.uniq[5] = (La == Lb && Lb == Lc && Lc == Ld) ? count(true, true, true) : 0;
}

// Integral store: the share of one job that rank `rank` of `n` evaluates when the launch deals flat units by U = rank (mod n) and the job's
// nwi work items form the units unit0 .. unit0 + ceil(nwi / chunk) - 1 (shell4_store_row): rows to allocate (owned units x chunk), work items
// among them (the last unit may be partial) and ubase = (first owned unit) / n.
struct StoreShare { long long rows = 0, items = 0, ubase = 0; };
inline StoreShare shell4_store_share(long long nwi, int chunk, long long unit0, int rank, int n) {
    StoreShare S;
    const long long nunits = (nwi + chunk - 1) / chunk, end = unit0 + nunits;
    const long long first = unit0 + ((rank - unit0 % n) % n + n) % n;
    S.ubase = first / n;
    if (first >= end) return S;
    const long long owned = (end - 1 - first) / n + 1;
    S.rows = owned * chunk;
    S.items = S.rows;
    if ((end - 1 - first) % n == 0) S.items -= nunits * chunk - nwi;      // the job's last unit is this rank's and is partial
    return S;
}

// View of the tables with the given base pointers (host vectors for the CPU test build, device copies for the GPU).
template <class PtrOf>
inline Class4Dev class4_view(const Class4Host& C, PtrOf ptr) {
    Class4Dev V;
    V.nchunk = (int)C.chunk_row0.size() - 1; V.nwork = C.nwork; V.nstage = C.nstage; V.nkst = C.nkst; V.itmax = C.itmax; V.zrow = C.zrow;
    V.ssize = C.ssize; V.nbeta = C.nbeta; V.ngamma = C.ngamma;
    V.n_rt = (int)C.t_rt.size(); V.n_xy = (int)C.t_xy.size(); V.n_u = (int)C.t_u.size() / 2;
    V.t_rt = ptr(C.t_rt); V.t_xy = ptr(C.t_xy); V.t_u = ptr(C.t_u); V.t_s = ptr(C.t_s);
    V.chunk_s0 = ptr(C.chunk_s0); V.p4 = ptr(C.p4); V.chunk_t0 = ptr(C.chunk_t0); V.chunk_ni = ptr(C.chunk_ni);
    V.ntab = C.ntab; V.tabs = ptr(C.tabs); V.jbrow_off = C.jbrow_off; V.jgcol_off = C.jgcol_off; V.jinfo_off = C.jinfo_off;
    for (int s = 0; s < 4; ++s) {
        for (int g = 0; g < 8; ++g) V.pgofs[s][g] = C.pgofs[s][g];
        for (int g = 0; g < 4; ++g) V.gsz[s][g] = C.gsz[s][g];
        V.ncols[s] = C.ncols[s]; V.pgoff[s] = C.pgoff[s]; V.kind[s] = C.kind[s];
    }
    for (int i = 0; i < 64; ++i) V.plan[i] = C.plan[i];
    V.nterm2 = C.nterm2; V.terms = ptr(C.terms); V.tptr = ptr(C.tptr);
    V.wfl = ptr(C.wfl); V.wlist = ptr(C.wlist); V.nwlist = (int)C.wlist.size(); V.nout_sm = C.nterm2 > 0 ? 0 : C.nwork;
    V.acc = ptr(C.acc); V.pmap = ptr(C.pmap); V.omap = ptr(C.omap);
    V.jst_ptr = ptr(C.jst_ptr); V.jst_list = ptr(C.jst_list); V.jflush = ptr(C.jflush); V.njfl = (int)C.jflush.size();
    V.nfill = (int)C.fill.size() / 2; V.fill = ptr(C.fill); V.chunk_f0 = ptr(C.chunk_f0); V.fperm = ptr(C.fperm);
    V.nint = C.nint; V.canon = ptr(C.canon); V.chunk_c0 = ptr(C.chunk_c0);
    return V;
}

}  // namespace tuna
