// shell4.cuh — shell-quartet engine, generation 4 (direct J/K on a z-axis diatomic; the headline kernel of round 2).
//
// Same mathematics and the same phases 0-3 as shell_jk.cuh (Boys values -> R^n_w and the x/y convolution table -> ket z
// contraction U -> bra z contraction S); replaces, at shell granularity, the primitive-quartet evaluation of
// TUNA/tuna_integrals/tuna_integral.pyx:1142-1253 and the quartet driver :1312-1342, and digests straight into J/K
// (TUNA/tuna_scf.py:27-72) so that no N^4 tensor exists.  What changed against the round-1 engine (streamed term tables), and why (ncu, profiles/r02a_*):
//   * the streamed per-class term tables of the digestion are gone.  The integral buffer of a chunk is laid out as
//       slot(beta, gamma) = Rb[beta] + Cg[gamma]      beta = bra pair function (ax+bx, ay+by, az, bz), gamma likewise for the ket,
//     rows grouped by x/y parity class so that a row holds exactly the allowed gammas.  Every K accumulator walks
//     (other bra component) x (other ket component) with two small shared-memory tables (components sorted by parity group, the
//     inner group padded to pairs whose staged density is zero); J accumulators are contiguous row / strided column dot
//     products.  The round-1 engine streamed 4-8 bytes of table per FMA from L2 (the variant with half the instructions and twice the
//     table bytes was SLOWER, profiles/r02a_variants.log).
//   * integral assembly is tiled over two z combinations that share the x/y operands (kept in registers, m' loop unrolled per
//     trip count), and S is only formed for (lz12, lz34) blocks of even total parity (the others never feed an integral).
//   * per-quartet bookkeeping (item decode, prefactor, record staging) is done once per quartet instead of once per lane.
// The body is written against a Policy: DevPolicy<G> is the sm_100a kernel, HostPolicy the CPU unit-test build.
#pragma once
#include "shell_jk.cuh"

namespace tuna {

constexpr unsigned S4_ABSENT = 0xffffffffu;

// One K block: Out[u][v] += sum_{s,t} It[Rb(u,s) + Cg(v,t)] * Pst[s][t]   (u,s = the two bra components, v,t = the two ket components)
struct Kind4 {
    int bra_tab, ket_tab;      // word offsets of the table rows  T[u][s''] (slot of the bra pair function) and T[v][t''] in the table area
    int bra_pitch, ket_pitch;
    int inner_ket;             // 1: t is the inner loop, 0: s is
    int pbase;                 // first staged density entry of the block; entry (outer'', inner'') at pbase + outer'' * pad_inner + inner''
    int pad_inner;
    int oshell, ishell;        // shell (0..3 = A,B,C,D) of the outer / inner summation component
};

struct Class4Dev {
    int nchunk, nwork, nstage, nkst, itmax, zrow, ssize, nbeta, ngamma;
    int n_rt, n_xy, n_u;
    const unsigned *t_rt, *t_xy, *t_u, *t_s;      // phases 1-3 work lists (formats of ClassTablesDev)
    const int* chunk_s0;                          // [nchunk+1] first t_s entry of a chunk
    const unsigned* p4;                           // phase 4 tiles, four words each (below)
    const int* chunk_t0;                          // [nchunk+1] first tile of a chunk
    const int* chunk_ni;                          // [nchunk]   integral slots of a chunk
    // digestion tables, one set per chunk in global memory (slot units); the kernel keeps the current chunk's copy in shared
    // memory, multiplied by the slot size in bytes.  Layout of a set: T_AB[a][b''] | T_BA[b][a''] | T_CD[c][d''] | T_DC[d][c''] |
    // JbRow[nbeta] | JgCol[ngamma] | jinfo[4][4] = {first slot of the chunk's rows of parity class pc, rows, first Pb entry, 0}
    int ntab;
    const unsigned* tabs;                         // [nchunk][ntab]
    int jbrow_off, jgcol_off, jinfo_off;
    unsigned char pgofs[4][8];                    // per shell: padded-sorted offset of parity group g (entries 0..4)
    unsigned char gsz[4][4];                      //            components in group g
    int ncols[4], pgoff[4];                       // per parity class: gammas (= row length), first Pg staging entry
    Kind4 kind[4];                                // KAC, KAD, KBC, KBD
    // plan[(kind * 4 + g) * 4 + og] = first outer'' | outer count << 8 | first inner'' << 16 | inner pairs << 24 : the loop bounds of one
    // accumulator of parity g for outer parity group og (inner group g ^ og), 0 when either group is empty
    unsigned plan[64];
    // term mode (light classes, one chunk): the digestion of every accumulator is a list of (integral slot, staged density entry)
    // pairs kept in SHARED memory as byte offsets (built once per CTA from the 32-bit global list `terms`: slot | entry << 16, padded to
    // pairs with (zero row, entry 0)); tptr[w] = first pair | pairs << 20.  nterm2 = 0 selects the separable loops above.
    int nterm2;
    const unsigned* terms; const unsigned* tptr;
    // term mode flushes every accumulator straight from registers (a single-chunk class completes an accumulator in one pass): no
    // Out array, no flush phase.  wfl[w] = first | count << 16 | (1u << 31 for a Coulomb target), wlist = (row | col << 8) entries: one
    // entry for a K accumulator, the component pairs of the pair function for a J accumulator.
    const unsigned* wfl; const unsigned short* wlist; int nwlist;
    int nout_sm;                                  // accumulators kept in shared memory: nwork (separable mode) or 0 (term mode)
    // work list: acc[2 w] = kind | g << 4 | u << 8 | v << 16 for K (kind 0..3), kind | pc << 4 for J (4 = bra pair function,
    // 5 = ket pair function); acc[2 w + 1] = pair-function index for J.  Sorted by descending work; Out[] is in this order.
    const unsigned* acc;
    // staging / flush
    const unsigned short* pmap;                   // [nkst] staged K density entry -> (row | col << 8), row/col = shell_sel << 5 | component; 0xffff = pad (zero)
    const unsigned short* omap;                   // [nwork] K accumulator -> (row | col << 8); 0xffff for J accumulators
    const unsigned* jst_ptr; const unsigned short* jst_list;   // [ngamma + nbeta + 1] CSR of component pairs: Pg (staging order) then Pb
    const unsigned* jflush; int njfl;             // (row | col << 8) | work position << 16
    // fill mode (dense-tensor build, no densities): entry e of the class = {integral slot in its chunk's buffer, a | b << 8 | c << 16 | d << 24};
    // chunk_f0[ch] = first entry of chunk ch.  Built only for the fill job set (nfill = 0 otherwise).
    int nfill;
    const unsigned* fill; const int* chunk_f0;
    // scatter pass: fperm[(m - 1) * nfill + e'] = entry handled by position e' in mode m = 1, 2, 3 (entries ordered so that c, b or a is the
    // fastest index; mode 0 is the list order, d fastest): consecutive lanes then write neighbouring elements of the images of that mode
    const unsigned* fperm;
};

// Phase 4 tile (two z combinations zc, zc+1 of one x/y combination):
//   w0 = xoff | yoff << 16                                   XY rows of the x and y index pairs
//   w1 = soff | nzc << 16                                    S offset of (n = 0, zc) in the chunk slice; n stride
//   w2 = mx0 | mx1 << 4 | my0 << 8 | ny << 12 | cnt << 16    m range, first m', number of m', valid z combinations (1 or 2)
//   w3 = slot0 | slot1 << 16
struct Shell4Job {
    int La, Lb, Lc, Ld;
    int nppAB, nppCD;
    // Contracted classes: the nppAB * nppCD primitive quartets of a shell quartet are walked serially (phases 0-4 each), which leaves a
    // handful of lanes busy for thousands of iterations in classes like (ss|ss) of cc-pVQZ.  J and K are linear in the integrals, so a
    // shell quartet is split into `psplit` work items of `clen` consecutive bra primitive pairs each (clen * psplit >= nppAB); every item
    // digests and flushes its partial integrals on its own.  When every bra primitive pair already is its own work item and the ket still
    // has more than the target number of primitive pairs (an (s8 s8| s8 s8) quartet of cc-pVTZ walks 64 of them), the ket is split as well:
    // psplit = (bra chunks) * ksplit work items per shell quartet, item chunk c -> bra chunk c / ksplit, ket chunk c % ksplit (klen pairs).
    int psplit, clen, ksplit, klen;
    const int* bra_list; const int* ket_list;
    const long long* item_prefix;
    int nbra, same_class;
    int chunk;
    int dbg_skip;                   // development aid (TUNA_B200_DBG_SKIP): bit k set -> stage k is skipped (timing experiments only; 0 in production)
    long long nitems;
    double uniq[6];
    Class4Dev ct;
    // shared-memory layout of one group (offsets in doubles, each array interleaved over the NB quartets of a batch)
    int NS, NGZ, oB, oPz, oRt, oXY, oU, oS, oIt, oP, oOut, oRecA, oRecC, oAO, oPref, aostride, total;
    int tab_off, hdr_off;           // CTA-level areas behind the group slices (doubles): digestion tables, quartet headers
    // fill mode: work item wi writes its nfill (partial, unnormalised) integrals to fill_scratch[fill_base + wi * nfill + e]; the scatter
    // pass (shell4_fill_scatter) sums the primitive chunks of a shell quartet in a fixed order and writes the eight images
    double* fill_scratch;
    long long fill_base;
    const int* fill_pairs;          // [2 * nitems] (bra pair, ket pair) of every shell quartet of the job: the scatter pass decodes an item with one load
};

// Work items of a shell quartet for a target number of primitive quartets per item (0 = never split).
inline void shell4_split(Shell4Job& J, int target, bool split_ket) {
    const long long tot = (long long)J.nppAB * J.nppCD;
    int bra = (target > 0 && tot > target) ? (int)((tot + target - 1) / target) : 1;
    if (bra > J.nppAB) bra = J.nppAB;
    J.clen = (J.nppAB + bra - 1) / bra;
    bra = (J.nppAB + J.clen - 1) / J.clen;
    J.ksplit = 1; J.klen = J.nppCD;
    if (split_ket && target > 0 && J.clen == 1 && J.nppCD > target) {
        const int ks = (J.nppCD + target - 1) / target;
        J.klen = (J.nppCD + ks - 1) / ks;
        J.ksplit = (J.nppCD + J.klen - 1) / J.klen;
    }
    J.psplit = bra * J.ksplit;
}

inline void shell4_job_layout(Shell4Job& J, int nD) {
    const int Ltot = J.La + J.Lb + J.Lc + J.Ld, Lab = J.La + J.Lb, Lcd = J.Lc + J.Ld;
    J.NS = Ltot / 2 + 1;
    J.NGZ = (J.Lc + 1) * (J.Ld + 1);
    int o = 0;
    J.oB = o; o += Ltot + 1;
    J.oPz = o; o += Ltot + 1;
    J.oRt = o; o += (Ltot + 1) * J.NS;
    J.oXY = o; o += (Lab + 1) * (Lcd + 1) * J.NS;
    J.oU = o; o += (Lab + 1) * J.NGZ * J.NS;
    J.oS = o; o += J.ct.ssize + 2;                    // + slack read by the second lane of a half-filled tile
    J.oIt = o; o += J.ct.itmax + J.ct.zrow;           // integral slots, then the zero row absent bra rows point to
    J.oP = o; o += nD * J.ct.nstage;
    J.oOut = o; o += nD * J.ct.nout_sm;
    J.oRecA = o; o += sp_rec_size(J.La, J.Lb);
    J.oRecC = o; o += sp_rec_size(J.Lc, J.Ld);
    int lmax = J.La > J.Lc ? J.La : J.Lc;
    if (J.Lb > lmax) lmax = J.Lb;
    if (J.Ld > lmax) lmax = J.Ld;
    J.aostride = (lmax + 1) * (lmax + 2) / 2;
    J.oAO = o; o += (4 * J.aostride * (int)sizeof(int) + 7) / 8;
    J.oPref = o; o += 1;
    J.total = (o + 1) & ~1;
}

// Copy the digestion tables of chunk ch into the CTA's table area, scaled to byte offsets of an NB-interleaved slot.
// (Called by all threads of the CTA; the caller synchronises.)  Term mode: the area holds the term pairs as byte offsets relative
// to the group's slice (integral buffer / staged densities of density 0), then tptr.
template <int NB>
TUNA_HD void shell4_load_tables(const Class4Dev& CT, int ch, unsigned* tab, int tid, int nthreads, int oIt, int oP) {
    if (CT.nterm2 > 0) {
        for (int i = tid; i < 2 * CT.nterm2; i += nthreads) {
            const unsigned t = CT.terms[i];
            tab[2 * i] = ((unsigned)oIt + (t & 0xffffu)) * (unsigned)(NB * 8);
            tab[2 * i + 1] = ((unsigned)oP + (t >> 16)) * (unsigned)(NB * 8);
        }
        for (int i = tid; i < CT.nwork; i += nthreads) { tab[4 * CT.nterm2 + i] = CT.tptr[i]; tab[4 * CT.nterm2 + CT.nwork + i] = CT.wfl[i]; }
        unsigned short* wl = reinterpret_cast<unsigned short*>(tab + 4 * CT.nterm2 + 2 * CT.nwork);
        for (int i = tid; i < CT.nwlist; i += nthreads) wl[i] = CT.wlist[i];
        return;
    }
    const unsigned* src = CT.tabs + (size_t)ch * CT.ntab;
    const int nscaled = CT.jinfo_off;                 // everything before jinfo is a slot number (or S4_ABSENT)
    for (int i = tid; i < CT.ntab; i += nthreads) {
        unsigned v = src[i];
        if (i < nscaled) v = (v == S4_ABSENT) ? (unsigned)CT.itmax * (unsigned)(NB * 8) : v * (unsigned)(NB * 8);
        tab[i] = v;
    }
}

// N2 pairs of inner components of one outer component: integral addresses = base + table word, densities contiguous
template <int NB, int N2>
TUNA_HD void digest_row4(const char* base, const unsigned* irow, const double* pp, double* s0, double* s1) {
    unsigned c[2 * N2];
#pragma unroll
    for (int j = 0; j < N2; ++j) {
        const uint2 t = *reinterpret_cast<const uint2*>(irow + 2 * j);
        c[2 * j] = t.x; c[2 * j + 1] = t.y;
    }
#pragma unroll
    for (int j = 0; j < N2; ++j) {
        const QVec<NB> i0 = qld<NB>(reinterpret_cast<const double*>(base + c[2 * j])), i1 = qld<NB>(reinterpret_cast<const double*>(base + c[2 * j + 1]));
        const QVec<NB> p0 = qld<NB>(pp + 2 * j * NB), p1 = qld<NB>(pp + (2 * j + 1) * NB);
#pragma unroll
        for (int q = 0; q < NB; ++q) { s0[q] = fma(i0.v[q], p0.v[q], s0[q]); s1[q] = fma(i1.v[q], p1.v[q], s1[q]); }
    }
}

template <int NB, int NY>
TUNA_HD void assemble4(const double* xyx, const double* xyy, const double* sp0, int nzc, int mx0, int mx1, QVec<NB>& a0, QVec<NB>& a1) {
    QVec<NB> y[NY];
#pragma unroll
    for (int k = 0; k < NY; ++k) y[k] = qld<NB>(xyy + k * NB);
    for (int m = mx0; m <= mx1; ++m) {
        const double* sp = sp0 + m * nzc * NB;
        QVec<NB> t0, t1;
#pragma unroll
        for (int q = 0; q < NB; ++q) { t0.v[q] = 0.0; t1.v[q] = 0.0; }
#pragma unroll
        for (int k = 0; k < NY; ++k) {
            const QVec<NB> s0 = qld<NB>(sp + k * nzc * NB), s1 = qld<NB>(sp + (k * nzc + 1) * NB);
#pragma unroll
            for (int q = 0; q < NB; ++q) { t0.v[q] = fma(y[k].v[q], s0.v[q], t0.v[q]); t1.v[q] = fma(y[k].v[q], s1.v[q], t1.v[q]); }
        }
        const QVec<NB> x = qld<NB>(xyx + m * NB);
#pragma unroll
        for (int q = 0; q < NB; ++q) { a0.v[q] = fma(x.v[q], t0.v[q], a0.v[q]); a1.v[q] = fma(x.v[q], t1.v[q], a1.v[q]); }
    }
}

// Header of one quartet of a batch, decoded once (by one lane) before the group starts on it.
struct Quartet4 {
    int active, shA, shB, shC, shD, ia0;      // the four shells (A, B of the bra pair, C, D of the ket pair); first bra primitive pair of this work item | first ket primitive pair << 16
    double w;                                 // degeneracy weight
    long long recA, recC;                     // offsets of the pairs' first primitive records in ShellData::rec
    double pA, zA, pC, zC;                    // exponent sum and centre of the FIRST primitive pair of bra and ket (Boys argument without a memory round trip)
};

// NB shell quartets of one class processed together by one group of Pol::G lanes.  `tab` is the CTA's table area (shared memory on
// the device), holding the tables of chunk `tab_chunk` on entry (updated when the class has several chunks).
template <class Pol, int NB>
TUNA_HD void shell4_quartets(const Shell4Job& J, const ShellData& D, const Quartet4* hq, double* __restrict__ sm, unsigned* tab, int& tab_chunk,
                             int nD, const double* __restrict__ Pf, const double* __restrict__ Psym, double* Jf, double* Kf, int ncart) {
    const Class4Dev& CT = J.ct;
    const int La = J.La, Lb = J.Lb, Lc = J.Lc, Ld = J.Ld;
    const int Lab = La + Lb, Lcd = Lc + Ld, Ltot = Lab + Lcd, NS = J.NS, NGZ = J.NGZ;
    const int NTA = Lab / 2 + 1, NTC = Lcd / 2 + 1, nwork = CT.nwork, nstage = CT.nstage;
    const int aos = J.aostride;
    double* const Bq = sm + J.oB * NB; double* const pzq = sm + J.oPz * NB; double* const Rtq = sm + J.oRt * NB;
    double* const XYq = sm + J.oXY * NB; double* const Uq = sm + J.oU * NB; double* const Sq = sm + J.oS * NB;
    double* const Itq = sm + J.oIt * NB; double* const Pstq = sm + J.oP * NB; double* const Outq = sm + J.oOut * NB;
    double* const RAq = sm + J.oRecA * NB; double* const RCq = sm + J.oRecC * NB;
    int* const aoq = reinterpret_cast<int*>(sm + J.oAO * NB);          // [NB][4][aostride]
    double* const prefq = sm + J.oPref * NB;                           // [NB] prefactor of the current primitive quartet
    const int lane = Pol::lane();

    int qa = -1;
#pragma unroll
    for (int q = 0; q < NB; ++q) if (qa < 0 && hq[q].active) qa = q;
    if (qa < 0) return;                                  // uniform over the group: nothing to do (no barrier inside was reached)
    bool act[NB];
    const double* recA[NB]; const double* recC[NB];
    double w[NB];
#pragma unroll
    for (int q = 0; q < NB; ++q) {
        act[q] = hq[q].active != 0;
        const Quartet4& h = act[q] ? hq[q] : hq[qa];      // an inactive slot runs on the data of an active one with weight zero
        w[q] = act[q] ? h.w : 0.0;
        recA[q] = D.rec + h.recA; recC[q] = D.rec + h.recC;
        int* ao = aoq + q * 4 * aos;
        const int shA = h.shA, shB = h.shB, shC = h.shC, shD = h.shD;
        for (int x = lane; x < aos; x += Pol::G) {
            ao[x] = D.sh_ao[shA * SH_NCMAX + x]; ao[aos + x] = D.sh_ao[shB * SH_NCMAX + x];
            ao[2 * aos + x] = D.sh_ao[shC * SH_NCMAX + x]; ao[3 * aos + x] = D.sh_ao[shD * SH_NCMAX + x];
        }
    }
    Pol::sync();
    const int skip = J.dbg_skip;
    // ---- stage the density blocks (K blocks through pmap, pair-function sums through the CSR) and clear the accumulators
    for (int dn = 0; dn < nD && !(skip & 1); ++dn) {
        const double* P = Pf + (size_t)dn * ncart * ncart;
        const double* Ps = Psym + (size_t)dn * ncart * ncart;
        double* Pd = Pstq + dn * nstage * NB;
        for (int x = lane; x < CT.nkst; x += Pol::G) {
            const unsigned m = CT.pmap[x];
            QVec<NB> v;
            if (m == 0xffffu) {
#pragma unroll
                for (int q = 0; q < NB; ++q) v.v[q] = 0.0;
            } else {
                const int ri = ((m >> 5) & 3) * aos + (m & 31), ci = ((m >> 13) & 3) * aos + ((m >> 8) & 31);
#pragma unroll
                for (int q = 0; q < NB; ++q) {
                    const int* ao = aoq + q * 4 * aos;
                    v.v[q] = P[ao[ri] * ncart + ao[ci]];
                }
            }
            qst<NB>(Pd + x * NB, v);
        }
        for (int x = lane; x < CT.ngamma + CT.nbeta; x += Pol::G) {
            QVec<NB> v;
#pragma unroll
            for (int q = 0; q < NB; ++q) v.v[q] = 0.0;
            for (unsigned t = CT.jst_ptr[x]; t < CT.jst_ptr[x + 1]; ++t) {
                const unsigned m = CT.jst_list[t];
                const int ri = ((m >> 5) & 3) * aos + (m & 31), ci = ((m >> 13) & 3) * aos + ((m >> 8) & 31);
#pragma unroll
                for (int q = 0; q < NB; ++q) {
                    const int* ao = aoq + q * 4 * aos;
                    v.v[q] += Ps[ao[ri] * ncart + ao[ci]];
                }
            }
            qst<NB>(Pd + (CT.nkst + x) * NB, v);
        }
    }
    for (int x = lane; x < nD * CT.nout_sm * NB; x += Pol::G) Outq[x] = 0.0;
    for (int x = lane; x < CT.zrow * NB; x += Pol::G) Itq[CT.itmax * NB + x] = 0.0;
    const int recAsz = sp_rec_size(La, Lb), recCsz = sp_rec_size(Lc, Ld);
    const int oExA = SP_HDR + sp_ez_size(La, Lb), oExC = SP_HDR + sp_ez_size(Lc, Ld);
    const bool single = J.nppAB * J.nppCD == 1;
    const unsigned slotb = NB * 8;                        // bytes of one NB-interleaved slot

    for (int ch = 0; ch < CT.nchunk; ++ch) {
        const int t0 = CT.chunk_t0[ch], nt = CT.chunk_t0[ch + 1] - t0;
        if (!single) { for (int x = lane; x < CT.chunk_ni[ch] * NB; x += Pol::G) Itq[x] = 0.0; }
        if (tab_chunk != ch) {                            // (only classes with several chunks ever get here)
            Pol::sync_cta();
            shell4_load_tables<NB>(CT, ch, tab, Pol::cta_thread(), Pol::cta_threads(), J.oIt, J.oP);
            tab_chunk = ch;
            Pol::sync_cta();
        }
        for (int it = 0; it < J.clen; ++it)
            for (int kk = 0; kk < J.klen; ++kk) {
                // primitive pairs of every quartet of the batch (a work item past the last primitive pair runs on the last one with weight 0)
                int iaq[NB], icq[NB];
                bool pvalid[NB];
#pragma unroll
                for (int q = 0; q < NB; ++q) {
                    const int i0 = hq[act[q] ? q : qa].ia0;
                    const int ia = (i0 & 0xffff) + it, ic = (i0 >> 16) + kk;
                    pvalid[q] = ia < J.nppAB && ic < J.nppCD;
                    iaq[q] = ia < J.nppAB ? ia : J.nppAB - 1;
                    icq[q] = ic < J.nppCD ? ic : J.nppCD - 1;
                }
                // ---- phase 0: the two primitive shell-pair records, Boys values scaled by (-2 rho)^m, powers of PQz
#pragma unroll
                for (int q = 0; q < NB && !(skip & 2); ++q) {
                    const double* rA = recA[q] + iaq[q] * recAsz;
                    const double* rC = recC[q] + icq[q] * recCsz;
                    if (kk == 0) { for (int x = lane; x < recAsz; x += Pol::G) RAq[x * NB + q] = rA[x]; }
                    for (int x = lane; x < recCsz; x += Pol::G) RCq[x * NB + q] = rC[x];
                }
                for (int x = lane; x < NB * 32 && !(skip & 2); x += Pol::G) {
                    const int q = x >> 5, m = x & 31;
                    if (m <= Ltot) {
                        const double* rA = recA[0] + iaq[0] * recAsz;
                        const double* rC = recC[0] + icq[0] * recCsz;
                        int qs = act[0] ? 0 : qa, ia = iaq[0], ic = icq[0];
                        bool pv = pvalid[0];
#pragma unroll
                        for (int k = 1; k < NB; ++k) if (q == k) { rA = recA[k] + iaq[k] * recAsz; rC = recC[k] + icq[k] * recCsz; qs = act[k] ? k : qa; ia = iaq[k]; ic = icq[k]; pv = pvalid[k]; }
                        double p, qq, PQz;
                        if (ia == 0 && ic == 0) { p = hq[qs].pA; qq = hq[qs].pC; PQz = hq[qs].zA - hq[qs].zC; }
                        else { p = rA[0]; qq = rC[0]; PQz = rA[1] - rC[1]; }
                        const double pq = p + qq, rho = p * qq / pq;
                        const double f = boys_single(D.boys, m, rho * PQz * PQz);
                        double s = 1.0, z = 1.0;
                        for (int k = 0; k < m; ++k) { s *= -2.0 * rho; z *= PQz; }
                        Bq[m * NB + q] = f * s;
                        pzq[m * NB + q] = z;
                        // the prefactor of this primitive quartet, once per quartet (a division and a square root per lane would be
                        // a third of all instructions of the light classes); read back in phase 4, three barriers later
                        if (m == 0) {
                            double wq = w[0];
#pragma unroll
                            for (int k = 1; k < NB; ++k) if (q == k) wq = w[k];
                            prefq[q] = pv ? wq * rA[2] * rC[2] * 34.986836655249725 / (p * qq * sqrt(pq)) : 0.0;
                        }
                    }
                }
                Pol::sync();
                // ---- phase 1: R^n_w (closed form) and the x/y convolution table
                for (int i = lane; i < CT.n_rt && !(skip & 4); i += Pol::G) {
                    const unsigned e = CT.t_rt[i];
                    const int wv = (e >> 16) & 255, n = e >> 24;
                    QVec<NB> r;
#pragma unroll
                    for (int q = 0; q < NB; ++q) r.v[q] = 0.0;
                    for (int k = 0; 2 * k <= wv; ++k) {
                        const double h = D.herm[wv * HERM_STRIDE + k];
                        const QVec<NB> z = qld<NB>(pzq + (wv - 2 * k) * NB), b = qld<NB>(Bq + (n + wv - k) * NB);
#pragma unroll
                        for (int q = 0; q < NB; ++q) r.v[q] = fma(h * z.v[q], b.v[q], r.v[q]);
                    }
                    qst<NB>(Rtq + (e & 0xffffu) * NB, r);
                }
                for (int i = lane; i < CT.n_xy && !(skip & 4); i += Pol::G) {
                    const unsigned e = CT.t_xy[i];
                    const int n12 = (e >> 16) & 15, n34 = (e >> 20) & 15, m = e >> 24, px = n12 & 1;
                    const int tlo = (2 * m - n34 > px) ? 2 * m - n34 : px;
                    const int thi = (2 * m - px < n12) ? 2 * m - px : n12;
                    const double df = (n34 & 1) ? -odd_dfact(m) : odd_dfact(m);
                    const double* ExA = RAq + (oExA + n12 * NTA) * NB;
                    const double* ExC = RCq + (oExC + n34 * NTC) * NB;
                    QVec<NB> v;
#pragma unroll
                    for (int q = 0; q < NB; ++q) v.v[q] = 0.0;
                    for (int t = tlo; t <= thi; t += 2) {
                        const QVec<NB> a = qld<NB>(ExA + (t >> 1) * NB), c = qld<NB>(ExC + ((2 * m - t) >> 1) * NB);
#pragma unroll
                        for (int q = 0; q < NB; ++q) v.v[q] = fma(a.v[q], c.v[q], v.v[q]);
                    }
#pragma unroll
                    for (int q = 0; q < NB; ++q) v.v[q] *= df;
                    qst<NB>(XYq + (e & 0xffffu) * NB, v);
                }
                Pol::sync();
                // ---- phase 2: U[v][gz][n] = sum_phi (-1)^phi Ez_CD[gz][phi] R^n_{v+phi}   (the sign rides on the FMA)
                for (int i = lane; i < CT.n_u && !(skip & 8); i += Pol::G) {
                    const unsigned e0w = CT.t_u[2 * i], e1w = CT.t_u[2 * i + 1];
                    const int lz34 = e1w >> 16;
                    const double* e = RCq + (SP_HDR + (e1w & 0xffffu)) * NB;
                    const double* r = Rtq + (e0w >> 16) * NB;
                    QVec<NB> u;
#pragma unroll
                    for (int q = 0; q < NB; ++q) u.v[q] = 0.0;
                    for (int phi = 0; phi <= lz34; ++phi) {
                        const QVec<NB> ev = qld<NB>(e + phi * NB), rv = qld<NB>(r + phi * NS * NB);
                        if (phi & 1) {
#pragma unroll
                            for (int q = 0; q < NB; ++q) u.v[q] = fma(-ev.v[q], rv.v[q], u.v[q]);
                        } else {
#pragma unroll
                            for (int q = 0; q < NB; ++q) u.v[q] = fma(ev.v[q], rv.v[q], u.v[q]);
                        }
                    }
                    qst<NB>(Uq + (e0w & 0xffffu) * NB, u);
                }
                Pol::sync();
                // ---- phase 3: S[block][n][zc] = sum_v Ez_AB[az][bz][v] U[v][gz][n] for the chunk's bra z rows, even blocks only
                {
                    const int ustride = NGZ * NS;
                    for (int i = CT.chunk_s0[ch] + lane; i < CT.chunk_s0[ch + 1] && !(skip & 16); i += Pol::G) {
                        const unsigned e0w = CT.t_s[2 * i], e1w = CT.t_s[2 * i + 1];
                        const int lz12 = e1w >> 16;
                        const double* e = RAq + (SP_HDR + (e1w & 0xffffu)) * NB;
                        const double* u = Uq + (e0w >> 16) * NB;
                        QVec<NB> sacc;
#pragma unroll
                        for (int q = 0; q < NB; ++q) sacc.v[q] = 0.0;
                        for (int v = 0; v <= lz12; ++v) {
                            const QVec<NB> ev = qld<NB>(e + v * NB), uv = qld<NB>(u + v * ustride * NB);
#pragma unroll
                            for (int q = 0; q < NB; ++q) sacc.v[q] = fma(ev.v[q], uv.v[q], sacc.v[q]);
                        }
                        qst<NB>(Sq + (e0w & 0xffffu) * NB, sacc);
                    }
                }
                Pol::sync();
                // ---- phase 4: integral assembly, two z combinations per tile
                {
                    double pref[NB];
#pragma unroll
                    for (int q = 0; q < NB; ++q) pref[q] = prefq[q];
                    const uint4* p4 = reinterpret_cast<const uint4*>(CT.p4) + t0;
                    int e = lane;
                    uint4 nxt;
                    nxt.x = nxt.y = nxt.z = nxt.w = 0u;
                    if (skip & 32) e = nt;
                    if (e < nt) nxt = p4[e];
                    for (; e < nt; e += Pol::G) {
                        const uint4 tw = nxt;
                        if (e + Pol::G < nt) nxt = p4[e + Pol::G];
                        const int xo = tw.x & 0xffffu, yo = tw.x >> 16, so = tw.y & 0xffffu, nzc = tw.y >> 16;
                        const int mx0 = tw.z & 15, mx1 = (tw.z >> 4) & 15, my0 = (tw.z >> 8) & 15, ny = (tw.z >> 12) & 15, cnt = tw.z >> 16;
                        const double* xyx = XYq + xo * NB;
                        const double* xyy = XYq + (yo + my0) * NB;
                        const double* sp0 = Sq + (so + my0 * nzc) * NB;
                        QVec<NB> a0, a1;
#pragma unroll
                        for (int q = 0; q < NB; ++q) { a0.v[q] = 0.0; a1.v[q] = 0.0; }
                        switch (ny) {
                            case 1: assemble4<NB, 1>(xyx, xyy, sp0, nzc, mx0, mx1, a0, a1); break;
                            case 2: assemble4<NB, 2>(xyx, xyy, sp0, nzc, mx0, mx1, a0, a1); break;
                            case 3: assemble4<NB, 3>(xyx, xyy, sp0, nzc, mx0, mx1, a0, a1); break;
                            case 4: assemble4<NB, 4>(xyx, xyy, sp0, nzc, mx0, mx1, a0, a1); break;
                            default:
                                for (int m = mx0; m <= mx1; ++m) {
                                    const double* sp = sp0 + m * nzc * NB;
                                    QVec<NB> t0v, t1v;
#pragma unroll
                                    for (int q = 0; q < NB; ++q) { t0v.v[q] = 0.0; t1v.v[q] = 0.0; }
                                    for (int k = 0; k < ny; ++k) {
                                        const QVec<NB> y = qld<NB>(xyy + k * NB), s0 = qld<NB>(sp + k * nzc * NB), s1 = qld<NB>(sp + (k * nzc + 1) * NB);
#pragma unroll
                                        for (int q = 0; q < NB; ++q) { t0v.v[q] = fma(y.v[q], s0.v[q], t0v.v[q]); t1v.v[q] = fma(y.v[q], s1.v[q], t1v.v[q]); }
                                    }
                                    const QVec<NB> x = qld<NB>(xyx + m * NB);
#pragma unroll
                                    for (int q = 0; q < NB; ++q) { a0.v[q] = fma(x.v[q], t0v.v[q], a0.v[q]); a1.v[q] = fma(x.v[q], t1v.v[q], a1.v[q]); }
                                }
                        }
                        double* i0 = Itq + (tw.w & 0xffffu) * NB;
                        double* i1 = Itq + (tw.w >> 16) * NB;
                        if (single) {
#pragma unroll
                            for (int q = 0; q < NB; ++q) { a0.v[q] *= pref[q]; a1.v[q] *= pref[q]; }
                            qst<NB>(i0, a0);
                            if (cnt > 1) qst<NB>(i1, a1);
                        } else {
                            QVec<NB> it = qld<NB>(i0);
#pragma unroll
                            for (int q = 0; q < NB; ++q) it.v[q] = fma(pref[q], a0.v[q], it.v[q]);
                            qst<NB>(i0, it);
                            if (cnt > 1) {
                                it = qld<NB>(i1);
#pragma unroll
                                for (int q = 0; q < NB; ++q) it.v[q] = fma(pref[q], a1.v[q], it.v[q]);
                                qst<NB>(i1, it);
                            }
                        }
                    }
                }
            }
        Pol::sync();
        // ---- phase 5: digestion of the chunk, one accumulator per lane; all addressing from the shared-memory tables
        if (J.fill_scratch) {
            // fill mode: the chunk's integrals go to the work items' scratch rows in list order (coalesced over the lanes)
            const int f0 = CT.chunk_f0[ch], nf = CT.chunk_f0[ch + 1] - f0;
            double* const row = J.fill_scratch + J.fill_base + Pol::work_item_of(J, hq) * (long long)CT.nfill + f0;      // hq[q] is work item work_item_of + q
            for (int e = lane; e < nf; e += Pol::G) {
                const QVec<NB> v = qld<NB>(Itq + CT.fill[2 * (f0 + e)] * NB);
#pragma unroll
                for (int q = 0; q < NB; ++q) if (act[q]) row[(long long)q * CT.nfill + e] = v.v[q];
            }
        } else if (skip & 64) {
        } else if (CT.nterm2 > 0) {
            // term mode: (integral, density) byte-offset pairs of the accumulator, two terms per 16-byte shared load
            const char* const smB = reinterpret_cast<const char*>(sm);
            const unsigned* tptr = tab + 4 * CT.nterm2;
            const unsigned* wfl = tptr + nwork;
            const unsigned short* wlist = reinterpret_cast<const unsigned short*>(wfl + nwork);
            for (int wi = lane; wi < nwork; wi += Pol::G) {
                const unsigned tp = tptr[wi];
                const unsigned n2 = tp >> 20;
                if (n2 == 0) continue;
                const uint4* tl = reinterpret_cast<const uint4*>(tab) + (tp & 0xfffffu);
                const unsigned fl = wfl[wi];
                for (int dn = 0; dn < nD; ++dn) {
                    const char* const pB = smB + dn * nstage * (NB * 8);
                    double s0[NB], s1[NB];
#pragma unroll
                    for (int q = 0; q < NB; ++q) { s0[q] = 0.0; s1[q] = 0.0; }
                    unsigned t = 0;
                    for (; t + 1 < n2; t += 2) {
                        const uint4 ta = tl[t], tb = tl[t + 1];
                        const QVec<NB> i0 = qld<NB>(reinterpret_cast<const double*>(smB + ta.x)), p0 = qld<NB>(reinterpret_cast<const double*>(pB + ta.y));
                        const QVec<NB> i1 = qld<NB>(reinterpret_cast<const double*>(smB + ta.z)), p1 = qld<NB>(reinterpret_cast<const double*>(pB + ta.w));
                        const QVec<NB> i2 = qld<NB>(reinterpret_cast<const double*>(smB + tb.x)), p2 = qld<NB>(reinterpret_cast<const double*>(pB + tb.y));
                        const QVec<NB> i3 = qld<NB>(reinterpret_cast<const double*>(smB + tb.z)), p3 = qld<NB>(reinterpret_cast<const double*>(pB + tb.w));
#pragma unroll
                        for (int q = 0; q < NB; ++q) {
                            s0[q] = fma(i0.v[q], p0.v[q], s0[q]); s1[q] = fma(i1.v[q], p1.v[q], s1[q]);
                            s0[q] = fma(i2.v[q], p2.v[q], s0[q]); s1[q] = fma(i3.v[q], p3.v[q], s1[q]);
                        }
                    }
                    if (t < n2) {
                        const uint4 ta = tl[t];
                        const QVec<NB> i0 = qld<NB>(reinterpret_cast<const double*>(smB + ta.x)), p0 = qld<NB>(reinterpret_cast<const double*>(pB + ta.y));
                        const QVec<NB> i1 = qld<NB>(reinterpret_cast<const double*>(smB + ta.z)), p1 = qld<NB>(reinterpret_cast<const double*>(pB + ta.w));
#pragma unroll
                        for (int q = 0; q < NB; ++q) { s0[q] = fma(i0.v[q], p0.v[q], s0[q]); s1[q] = fma(i1.v[q], p1.v[q], s1[q]); }
                    }
                    if (skip & 128) continue;
                    double* const M = ((fl >> 31) ? Jf : Kf) + (size_t)dn * ncart * ncart;
                    const unsigned f0 = fl & 0xffffu, f1 = f0 + ((fl >> 16) & 0x7fffu);
                    for (unsigned e = f0; e < f1; ++e) {
                        const unsigned m = wlist[e];
                        const int ri = ((m >> 5) & 3) * aos + (m & 31), ci = ((m >> 13) & 3) * aos + ((m >> 8) & 31);
#pragma unroll
                        for (int q = 0; q < NB; ++q) {
                            const double v = s0[q] + s1[q];
                            if (!act[q] || v == 0.0) continue;
                            const int* ao = aoq + q * 4 * aos;
                            Pol::accumulate(M, ao[ri] * ncart + ao[ci], v, D.fix_lo);
                        }
                    }
                }
            }
        } else {
            const char* const ItB = reinterpret_cast<const char*>(Itq);
            const unsigned* jinfo = tab + CT.jinfo_off;
            int wi = lane;
            unsigned nx0 = 0u, nx1 = 0u;
            if (wi < nwork) { nx0 = CT.acc[2 * wi]; nx1 = CT.acc[2 * wi + 1]; }
            for (; wi < nwork; wi += Pol::G) {
                const unsigned a0w = nx0, a1w = nx1;
                if (wi + Pol::G < nwork) { nx0 = CT.acc[2 * (wi + Pol::G)]; nx1 = CT.acc[2 * (wi + Pol::G) + 1]; }
                const int kd = a0w & 15;
                for (int dn = 0; dn < nD; ++dn) {
                    const double* Pd = Pstq + dn * nstage * NB;
                    double s0[NB], s1[NB];
#pragma unroll
                    for (int q = 0; q < NB; ++q) { s0[q] = 0.0; s1[q] = 0.0; }
                    if (kd < 4) {
                        const Kind4& K = CT.kind[kd];
                        const int g = (a0w >> 4) & 3, u = (a0w >> 8) & 255, v = (a0w >> 16) & 255;
                        const int ik = K.inner_ket, padi = K.pad_inner;
                        const unsigned* brow = tab + K.bra_tab + u * K.bra_pitch;
                        const unsigned* krow = tab + K.ket_tab + v * K.ket_pitch;
                        const unsigned* orow = ik ? brow : krow;
                        const unsigned* irow = ik ? krow : brow;
                        const double* Pk = Pd + K.pbase * NB;
                        const unsigned* plan = CT.plan + (kd * 4 + g) * 4;
#pragma unroll 1
                        for (int og = 0; og < 4; ++og) {
                            const unsigned pl = plan[og];
                            if (pl == 0u) continue;
                            const int ob = pl & 255, on = (pl >> 8) & 255, ib = (pl >> 16) & 255, n2 = pl >> 24;
                            const unsigned* ir = irow + ib;
                            const double* pp = Pk + (ob * padi + ib) * NB;
                            const unsigned* op = orow + ob;
                            if (n2 == 3) {
#pragma unroll 1
                                for (int o = 0; o < on; ++o, pp += padi * NB) digest_row4<NB, 3>(ItB + op[o], ir, pp, s0, s1);
                            } else if (n2 == 2) {
#pragma unroll 1
                                for (int o = 0; o < on; ++o, pp += padi * NB) digest_row4<NB, 2>(ItB + op[o], ir, pp, s0, s1);
                            } else if (n2 == 1) {
#pragma unroll 1
                                for (int o = 0; o < on; ++o, pp += padi * NB) digest_row4<NB, 1>(ItB + op[o], ir, pp, s0, s1);
                            } else {
                                for (int o = 0; o < on; ++o, pp += padi * NB) {
                                    const char* base = ItB + op[o];
                                    for (int i = 0; i < n2; ++i) digest_row4<NB, 1>(base, ir + 2 * i, pp + 2 * i * NB, s0, s1);
                                }
                            }
                        }
                    } else if (kd == 4) {
                        // bra pair function beta: contiguous row of the chunk's buffer against the staged ket densities of its class
                        const unsigned row = tab[CT.jbrow_off + a1w];
                        const int pc = (a0w >> 4) & 3;
                        if (row != (unsigned)CT.itmax * slotb) {
                            const double* ip = reinterpret_cast<const double*>(ItB + row);
                            const double* pp = Pd + (CT.nkst + CT.pgoff[pc]) * NB;
                            const int n = CT.ncols[pc];
                            int k = 0;
                            for (; k + 3 < n; k += 4) {
                                const QVec<NB> i0 = qld<NB>(ip + k * NB), i1 = qld<NB>(ip + (k + 1) * NB), i2 = qld<NB>(ip + (k + 2) * NB), i3 = qld<NB>(ip + (k + 3) * NB);
                                const QVec<NB> p0 = qld<NB>(pp + k * NB), p1 = qld<NB>(pp + (k + 1) * NB), p2 = qld<NB>(pp + (k + 2) * NB), p3 = qld<NB>(pp + (k + 3) * NB);
#pragma unroll
                                for (int q = 0; q < NB; ++q) {
                                    s0[q] = fma(i0.v[q], p0.v[q], s0[q]); s1[q] = fma(i1.v[q], p1.v[q], s1[q]);
                                    s0[q] = fma(i2.v[q], p2.v[q], s0[q]); s1[q] = fma(i3.v[q], p3.v[q], s1[q]);
                                }
                            }
                            for (; k < n; ++k) {
                                const QVec<NB> i0 = qld<NB>(ip + k * NB), p0 = qld<NB>(pp + k * NB);
#pragma unroll
                                for (int q = 0; q < NB; ++q) s0[q] = fma(i0.v[q], p0.v[q], s0[q]);
                            }
                        }
                    } else {
                        // ket pair function gamma: column of the chunk's rows of its parity class against the staged bra densities
                        const int pc = (a0w >> 4) & 3;
                        const unsigned col = tab[CT.jgcol_off + a1w];
                        const unsigned row0 = jinfo[4 * pc] * slotb, nrows = jinfo[4 * pc + 1], pb0 = jinfo[4 * pc + 2];
                        const unsigned stride = (unsigned)CT.ncols[pc] * slotb;
                        const char* ip = ItB + row0 + col;
                        const double* pp = Pd + (CT.nkst + CT.ngamma + pb0) * NB;
                        unsigned r = 0;
                        for (; r + 1 < nrows; r += 2, ip += 2 * stride, pp += 2 * NB) {
                            const QVec<NB> i0 = qld<NB>(reinterpret_cast<const double*>(ip)), i1 = qld<NB>(reinterpret_cast<const double*>(ip + stride));
                            const QVec<NB> p0 = qld<NB>(pp), p1 = qld<NB>(pp + NB);
#pragma unroll
                            for (int q = 0; q < NB; ++q) { s0[q] = fma(i0.v[q], p0.v[q], s0[q]); s1[q] = fma(i1.v[q], p1.v[q], s1[q]); }
                        }
                        if (r < nrows) {
                            const QVec<NB> i0 = qld<NB>(reinterpret_cast<const double*>(ip)), p0 = qld<NB>(pp);
#pragma unroll
                            for (int q = 0; q < NB; ++q) s0[q] = fma(i0.v[q], p0.v[q], s0[q]);
                        }
                    }
                    QVec<NB> out = qld<NB>(Outq + (dn * nwork + wi) * NB);
#pragma unroll
                    for (int q = 0; q < NB; ++q) out.v[q] += s0[q] + s1[q];
                    qst<NB>(Outq + (dn * nwork + wi) * NB, out);
                }
            }
        }
        Pol::sync();
    }
    // ---- flush the shell blocks (separable mode; term mode has flushed from registers)
    for (int dn = 0; dn < nD && !(skip & 128) && CT.nterm2 == 0; ++dn) {
        double* Kd = Kf + (size_t)dn * ncart * ncart;
        double* Jd = Jf + (size_t)dn * ncart * ncart;
        for (int x = lane; x < nwork; x += Pol::G) {
            const unsigned m = CT.omap[x];
            if (m == 0xffffu) continue;                    // pair-function accumulator: expanded below
            const int ri = ((m >> 5) & 3) * aos + (m & 31), ci = ((m >> 13) & 3) * aos + ((m >> 8) & 31);
            const QVec<NB> v = qld<NB>(Outq + (dn * nwork + x) * NB);
#pragma unroll
            for (int q = 0; q < NB; ++q) {
                if (!act[q] || v.v[q] == 0.0) continue;
                const int* ao = aoq + q * 4 * aos;
                Pol::accumulate(Kd, ao[ri] * ncart + ao[ci], v.v[q], D.fix_lo);
            }
        }
        for (int x = lane; x < CT.njfl; x += Pol::G) {
            const unsigned e = CT.jflush[x], m = e & 0xffffu;
            const int ri = ((m >> 5) & 3) * aos + (m & 31), ci = ((m >> 13) & 3) * aos + ((m >> 8) & 31);
            const QVec<NB> v = qld<NB>(Outq + (dn * nwork + (e >> 16)) * NB);
#pragma unroll
            for (int q = 0; q < NB; ++q) {
                if (!act[q] || v.v[q] == 0.0) continue;
                const int* ao = aoq + q * 4 * aos;
                Pol::accumulate(Jd, ao[ri] * ncart + ao[ci], v.v[q], D.fix_lo);
            }
        }
    }
    Pol::sync();
}

// Fill mode, second pass: position ep of shell quartet `item` of a job in mode m.  Sums the primitive chunks in a fixed order (bitwise
// reproducible, no atomics), applies the component norms and writes the canonical value to the two images of the dense n^4 tensor whose
// LAST index is the component the mode's entry order varies fastest (m = 0: d, 1: c, 2: b, 3: a), so that the lanes of a warp write
// neighbouring elements; the four modes together write all eight images.  Component quartets that another entry of the same block
// represents (A = B with b > a, C = D with d > c, bra pair = ket pair with (c, d) > (a, b)) are skipped, so every element of the tensor
// has one value.  (Parity-forbidden elements stay zero from the memset.)
TUNA_HD void shell4_fill_scatter(const Shell4Job& J, const ShellData& D, long long item, int ep, int mode, const double* __restrict__ fnorm,
                                 double* __restrict__ out, long long n) {
    const int nf = J.ct.nfill;
    const int e = mode == 0 ? ep : (int)J.ct.fperm[(size_t)(mode - 1) * nf + ep];
    const int pab = J.fill_pairs[2 * item], pcd = J.fill_pairs[2 * item + 1];
    const int shA = D.pairA[pab], shB = D.pairB[pab], shC = D.pairA[pcd], shD = D.pairB[pcd];
    const unsigned m = J.ct.fill[2 * e + 1];
    const int a = m & 255, b = (m >> 8) & 255, c = (m >> 16) & 255, d = m >> 24;
    if (shA == shB && b > a) return;
    if (shC == shD && d > c) return;
    if (pab == pcd && (c > a || (c == a && d > b))) return;
    const double* s = J.fill_scratch + J.fill_base + item * J.psplit * nf + e;
    double v = 0.0;
    for (int pc = 0; pc < J.psplit; ++pc) v += s[(long long)pc * nf];
    const long long i = D.sh_ao[shA * SH_NCMAX + a], j = D.sh_ao[shB * SH_NCMAX + b], k = D.sh_ao[shC * SH_NCMAX + c], l = D.sh_ao[shD * SH_NCMAX + d];
    v *= fnorm[i] * fnorm[j] * fnorm[k] * fnorm[l];
    const long long n2 = n * n, n3 = n2 * n;
    switch (mode) {
        case 0: out[i * n3 + j * n2 + k * n + l] = v; out[j * n3 + i * n2 + k * n + l] = v; break;
        case 1: out[i * n3 + j * n2 + l * n + k] = v; out[j * n3 + i * n2 + l * n + k] = v; break;
        case 2: out[k * n3 + l * n2 + i * n + j] = v; out[l * n3 + k * n2 + i * n + j] = v; break;
        default: out[k * n3 + l * n2 + j * n + i] = v; out[l * n3 + k * n2 + j * n + i] = v; break;
    }
}

// Per-shell Cartesian->spherical blocks (SphShells of shell_host.hpp, on the device)
struct SphData {
    const int* nsph; const int* sph; const int* uoff; const double* u; const int* par;
};

TUNA_HD int sph_ncart(int L) { return (L + 1) * (L + 2) / 2; }

// Spherical fill, second pass: shell quartet `item` of a job straight into the spherical tensor (dimension n).  The CTA
//   1. sums the primitive chunks of every fill entry in the order of shell4_fill_scatter, applies the component norms and stores the
//      Cartesian block E[a][b][c][d] in `cart` (parity-forbidden entries zero);
//   2. for every spherical function p of A: X[b][c][d] = sum_a U_A[p][a] E, then Y[q][c][d] = sum_b U_B[q][b] X, X[q][r][d] = sum_c U_C[r][c] Y,
//      and each (q, r, s) sums over d and writes its value to the eight images.
// Every sum runs in a fixed order (bitwise reproducible, no atomics).  Spherical quartets that another element of the same block represents
// (A = B with q > p, C = D with s > r, bra pair = ket pair with (r, s) > (p, q)) are skipped, so every element has one value; a quartet whose
// parities do not cancel is written as an exact zero.  cart holds nA nB nC nD doubles, X and Y nB nC nD each.
template <class Pol>
TUNA_HD void shell4_fill_sph(const Shell4Job& J, const ShellData& D, const SphData& Y, long long item, const double* __restrict__ fnorm,
                             double* __restrict__ cart, double* __restrict__ X, double* __restrict__ Yb, double* __restrict__ out, long long n) {
    const int tid = Pol::cta_thread(), nt = Pol::cta_threads();
    const int nf = J.ct.nfill;
    const int pab = J.fill_pairs[2 * item], pcd = J.fill_pairs[2 * item + 1];
    const int shA = D.pairA[pab], shB = D.pairB[pab], shC = D.pairA[pcd], shD = D.pairB[pcd];
    const int nA = sph_ncart(J.La), nB = sph_ncart(J.Lb), nC = sph_ncart(J.Lc), nD = sph_ncart(J.Ld);
    const int mA = Y.nsph[shA], mB = Y.nsph[shB], mC = Y.nsph[shC], mD = Y.nsph[shD];
    const double *uA = Y.u + Y.uoff[shA], *uB = Y.u + Y.uoff[shB], *uC = Y.u + Y.uoff[shC], *uD = Y.u + Y.uoff[shD];
    const int ncd = nC * nD, nbcd = nB * ncd;
    for (int x = tid; x < nA * nbcd; x += nt) cart[x] = 0.0;
    Pol::sync_cta();
    const double* s = J.fill_scratch + J.fill_base + item * J.psplit * nf;
    for (int e = tid; e < nf; e += nt) {
        const unsigned m = J.ct.fill[2 * e + 1];
        const int a = m & 255, b = (m >> 8) & 255, c = (m >> 16) & 255, d = m >> 24;
        double v = 0.0;
        for (int pc = 0; pc < J.psplit; ++pc) v += s[(long long)pc * nf + e];
        v *= fnorm[D.sh_ao[shA * SH_NCMAX + a]] * fnorm[D.sh_ao[shB * SH_NCMAX + b]] * fnorm[D.sh_ao[shC * SH_NCMAX + c]] * fnorm[D.sh_ao[shD * SH_NCMAX + d]];
        cart[a * nbcd + b * ncd + c * nD + d] = v;
    }
    Pol::sync_cta();
    const long long n2 = n * n, n3 = n2 * n;
    for (int p = 0; p < mA; ++p) {
        for (int x = tid; x < nbcd; x += nt) {
            double v = 0.0;
            for (int a = 0; a < nA; ++a) {
                const double u = uA[p * nA + a];
                if (u != 0.0) v = fma(u, cart[a * nbcd + x], v);
            }
            X[x] = v;
        }
        Pol::sync_cta();
        for (int x = tid; x < mB * ncd; x += nt) {
            const int q = x / ncd, cd = x - q * ncd;
            double v = 0.0;
            for (int b = 0; b < nB; ++b) {
                const double u = uB[q * nB + b];
                if (u != 0.0) v = fma(u, X[b * ncd + cd], v);
            }
            Yb[x] = v;
        }
        Pol::sync_cta();
        for (int x = tid; x < mB * mC * nD; x += nt) {
            const int qr = x / nD, d = x - qr * nD, q = qr / mC, r = qr - q * mC;
            double v = 0.0;
            for (int c = 0; c < nC; ++c) {
                const double u = uC[r * nC + c];
                if (u != 0.0) v = fma(u, Yb[(q * nC + c) * nD + d], v);
            }
            X[x] = v;
        }
        Pol::sync_cta();
        const long long P = Y.sph[shA * SH_NCMAX + p];
        for (int x = tid; x < mB * mC * mD; x += nt) {
            const int qr = x / mD, sd = x - qr * mD, q = qr / mC, r = qr - q * mC;
            if (shA == shB && q > p) continue;
            if (shC == shD && sd > r) continue;
            if (pab == pcd && (r > p || (r == p && sd > q))) continue;
            const long long Q = Y.sph[shB * SH_NCMAX + q], R = Y.sph[shC * SH_NCMAX + r], S = Y.sph[shD * SH_NCMAX + sd];
            double v = 0.0;
            if ((Y.par[P] ^ Y.par[Q] ^ Y.par[R] ^ Y.par[S]) == 0)
                for (int d = 0; d < nD; ++d) {
                    const double u = uD[sd * nD + d];
                    if (u != 0.0) v = fma(u, X[qr * nD + d], v);
                }
            out[P * n3 + Q * n2 + R * n + S] = v; out[Q * n3 + P * n2 + R * n + S] = v;
            out[P * n3 + Q * n2 + S * n + R] = v; out[Q * n3 + P * n2 + S * n + R] = v;
            out[R * n3 + S * n2 + P * n + Q] = v; out[S * n3 + R * n2 + P * n + Q] = v;
            out[R * n3 + S * n2 + Q * n + P] = v; out[S * n3 + R * n2 + Q * n + P] = v;
        }
        Pol::sync_cta();
    }
}

}  // namespace tuna
