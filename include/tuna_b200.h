/*
 * tuna_b200.h — C ABI of libtuna_b200.so: the B200 (sm_100a) provider for TUNA's SCF two-electron hot path.
 *
 * Drop-in boundary (SURVEY.md section 8b).  Each entry point names the reference interface it replaces;
 * paths are relative to h-brough/TUNA, "pyx" = TUNA/tuna_integrals/tuna_integral.pyx.
 *
 * Conventions: plain pointers and sizes only; every function returns an int status (0 = ok); no exceptions
 * or Python objects cross; the caller owns every host buffer; the library owns only memory behind the
 * opaque context; a context is not thread-safe; one context per (device, geometry, basis).  All matrices and
 * tensors are dense, C-order, IEEE double.  Entry points ending in _dev take DEVICE pointers and enqueue on
 * the context's stream without synchronising; all others take HOST pointers and return when the result is
 * in the caller's buffer.  There is no CPU fallback anywhere behind this header.
 */
#ifndef TUNA_B200_H
#define TUNA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct tuna_ctx tuna_ctx;

enum {
    TUNA_OK = 0,
    TUNA_ERR_ARG = 1,      /* bad argument            -> Python raises TunaError                       */
    TUNA_ERR_NOMEM = 2,    /* host or device OOM      -> MemoryError (pyx:1120, :1290 raise the same)   */
    TUNA_ERR_CUDA = 3,     /* CUDA runtime failure    -> TunaError                                      */
    TUNA_ERR_STATE = 4     /* call order / missing prerequisite -> TunaError                            */
};

/* Context life cycle.  `device` is the CUDA ordinal.  Uploads the Boys-function table. */
int tuna_ctx_create(int device, tuna_ctx** out);
int tuna_ctx_destroy(tuna_ctx* ctx);
const char* tuna_last_error(const tuna_ctx* ctx);
/* Use an externally owned cudaStream_t (e.g. torch.cuda.current_stream().cuda_stream); 0 = the context's own. */
int tuna_set_stream(tuna_ctx* ctx, void* cuda_stream);

/* The basis: one entry per CARTESIAN COMPONENT, exactly the list[Basis] the reference passes
 * (Basis: pyx:78-235; ordered as tuna_molecule.py:532-585 builds it).  coef_eff[k] = Basis.norm[k] * Basis.coefs[k]
 * (pyx:1070).  All centres must lie on the z axis (tuna_kernel.py:386-388); origins_z holds their z.
 * Builds the class-sorted AO-pair / primitive-pair table once (replaces pyx:1050-1128, :1300-1308). */
int tuna_set_basis(tuna_ctx* ctx, int ncart, const double* origins_z, const int32_t* lmn, const int32_t* nprim,
                   const int64_t* prim_offset, const double* exps, const double* coef_eff);

/* Cartesian -> spherical map U (nbf x ncart, row-major) = molecule.spherical_harmonic_transformation_matrix
 * (tuna_kernel.py:540-649).  Pass the identity for CARTHARM (tuna_kernel.py:481-483). */
int tuna_set_transform(tuna_ctx* ctx, int nbf, const double* U);

/* calculate_electron_repulsion_integrals (pyx:1267-1355): fill the dense Cartesian tensor ncart^4 on the device.  Contracted bases
 * that group into shells run the shell-quartet engine in fill mode plus a fixed-order scatter pass (bitwise reproducible); other
 * bases one thread per AO quartet (TUNA_B200_FILL_ENGINE=0/1 forces either).  Same tensor both ways: one value in all eight
 * symmetric images, exact zeros where x/y parity forbids the integral (pyx:1324-1327). */
int tuna_eri_fill_cart(tuna_ctx* ctx);
/* transform_to_spherical_harmonics, ERI part (tuna_kernel.py:504-523): (U (x) U) ERI (U (x) U)^T on the device.
 * keep_cart != 0 keeps the Cartesian tensor resident as well. */
int tuna_eri_cart_to_sph(tuna_ctx* ctx, int keep_cart);
/* The spherical tensor nbf^4 without the Cartesian one: the engine's fill mode, then a pass that rotates every shell quartet's
 * Cartesian block with the per-shell blocks of U and writes one value to all eight images (bitwise reproducible, exact parity zeros).
 * Needs tuna_set_basis and tuna_set_transform.  Leaves the spherical tensor resident as the stored tensor and no Cartesian tensor.
 * Bases the engine does not fill, a U that is not block-diagonal over the basis's shells, and the identity U run
 * tuna_eri_fill_cart + tuna_eri_cart_to_sph(ctx, 0) instead.  tuna_last_kernel_ms(0) times the fill. */
int tuna_eri_fill_sph(tuna_ctx* ctx);
/* Copy a resident tensor to the host: which = 0 Cartesian (ncart^4), 1 spherical (nbf^4). */
int tuna_eri_download(tuna_ctx* ctx, int which, double* host_out);
/* Adopt a dense n^4 tensor supplied by the caller as the stored tensor for tuna_jk_stored (a plain ndarray
 * handed to tuna_scf.calculate_coulomb_matrix / calculate_exchange_matrix). */
int tuna_eri_upload(tuna_ctx* ctx, int n, const double* host_in);
/* calculate_electron_repulsion_integral (pyx:1376-1414) for functions (i j | k l) of the current basis. */
int tuna_eri_single(tuna_ctx* ctx, int i, int j, int k, int l, double* out);
/* Schwarz factors Q_ij = sqrt((ij|ij)) as a dense ncart x ncart matrix (not in the reference; SURVEY.md 8d). */
int tuna_schwarz(tuna_ctx* ctx, double* host_out);

/* Stored-ERI Fock contraction: for each of nD densities P[d] (n x n),
 *   J[d]_ij = sum_kl (ij|kl) P_kl   (tuna_scf.calculate_coulomb_matrix,  tuna_scf.py:55-72)
 *   K[d]_ij = sum_kl (il|kj) P_kl   (tuna_scf.calculate_exchange_matrix, tuna_scf.py:27-44)
 * in ONE pass over the resident tensor.  J or K may be NULL.  n is the stored tensor's dimension. */
int tuna_jk_stored(tuna_ctx* ctx, int nD, const double* P, double* J, double* K);
int tuna_jk_stored_dev(tuna_ctx* ctx, int nD, const double* dP, double* dJ, double* dK);

/* Direct (integral-driven) Fock contraction: same J and K, in the basis of U (nbf x nbf matrices), never
 * materialising the tensor: 8-fold symmetry, Schwarz screening |Q_ij Q_kl| max|P| < tau skipped.
 * tau <= 0 disables screening.  tuna_jk_direct accepts any real P (a non-symmetric density is split into its symmetric and
 * antisymmetric parts: J[P] = J[S], K[P] = K[S] + K[A]).  tuna_jk_direct_dev REQUIRES symmetric densities and does not check:
 * it builds K = U (Kacc + Kacc^T) U^T, symmetric by construction, so for a non-symmetric P it silently drops K[A].  Callers with
 * possibly asymmetric densities (e.g. guess densities, asymmetric at ~1e-8) use tuna_jk_direct, or tuna_jk_direct_general_dev with
 * device buffers.
 * The cached quartet lists are pre-screened with tau / (1e3 max(1, max|P|)) for host densities; tuna_jk_direct_dev assumes max|P| <= ~10
 * (scale larger device densities down - J and K are linear in P; tuna_jk_direct_general_dev measures max|P| itself).  J and K are accumulated as 64-bit integers (order independent):
 * repeated builds are bitwise identical; |J|, |K| < 2^42 in the unnormalised Cartesian working basis is required. */
int tuna_jk_direct(tuna_ctx* ctx, int nD, const double* P, double* J, double* K, double tau);
int tuna_jk_direct_dev(tuna_ctx* ctx, int nD, const double* dP, double* dJ, double* dK, double tau);
/* tuna_jk_direct with DEVICE pointers (dP, dJ, dK on the context's device, enqueued on its stream): any real P, 1 <= nD <= 8, J or K may
 * be NULL.  max|P| and max|P - P^T| are taken on the device and read back (16 bytes, ONE stream synchronise, the only one of the call);
 * they set the pre-screening bound and decide the symmetric / antisymmetric split exactly as tuna_jk_direct does on the host, and the split
 * and the sum K[S] + K[A] run on the device with the host's arithmetic.  J and K are bitwise identical to tuna_jk_direct for the same P,
 * tau, shard and integral store state.  Everything after the read-back is enqueued without a further synchronise. */
int tuna_jk_direct_general_dev(tuna_ctx* ctx, int nD, const double* dP, double* dJ, double* dK, double tau);
/* Multi-GPU sharding of the quartet list for tuna_jk_direct*: this context evaluates only its share and
 * returns PARTIAL J/K, to be summed over ranks by the caller (one all-reduce per build, SURVEY.md 8e). */
int tuna_set_shard(tuna_ctx* ctx, int rank, int nranks);
/* Direct J/K of ONE Fock build spread over nctx contexts on pairwise distinct devices of this process: same basis and transform in
 * every context, ctxs[r] sharded as (r, nctx) with tuna_set_shard.  Each rank accumulates its share of the quartets on its own device
 * (enqueued from one host thread per device, all joined before the call returns); the 64-bit integer accumulators of all ranks are
 * pulled to ctxs[0]'s device and summed there before the conversion to FP64, so J and K are bitwise identical to tuna_jk_direct /
 * tuna_jk_direct_dev on one context (within FP64 round-off for bases that run the per-component kernel).  nctx == 1 is tuna_jk_direct.
 * TUNA_ERR_ARG: nctx < 1, a null or repeated context, two contexts on one device.  TUNA_ERR_STATE: a context with a different basis or
 * transform (ncart, nbf, checksums of the arrays given to tuna_set_basis / tuna_set_transform) or a shard other than (r, nctx).
 * Errors are reported through tuna_last_error(ctxs[0]), the failing rank named. */
int tuna_jk_direct_group(tuna_ctx* const* ctxs, int nctx, int nD, const double* P, double* J, double* K, double tau);
/* dP, dJ, dK on ctxs[0]'s device, enqueued on ctxs[0]'s stream; symmetric densities only, as tuna_jk_direct_dev (any real P:
 * tuna_jk_direct_group_general_dev). */
int tuna_jk_direct_group_dev(tuna_ctx* const* ctxs, int nctx, int nD, const double* dP, double* dJ, double* dK, double tau);
/* tuna_jk_direct_group with DEVICE pointers on ctxs[0]'s device, as tuna_jk_direct_general_dev: the scan, its read-back (one synchronise of
 * ctxs[0]'s stream), the split and K[S] + K[A] run on ctxs[0].  Bitwise identical to tuna_jk_direct_group and to tuna_jk_direct on one
 * context; the group's errors are those of tuna_jk_direct_group. */
int tuna_jk_direct_group_general_dev(tuna_ctx* const* ctxs, int nctx, int nD, const double* dP, double* dJ, double* dK, double tau);
/* Semi-direct J/K: keep the shell-quartet engine's contracted integrals of whole class jobs in device memory, up to budget_bytes
 * (0, the default, = off), and replay them in later tuna_jk_direct* / tuna_jk_direct_group* builds instead of evaluating them again.
 * The first build after the store is set (or dropped) plans it and fills it while it runs; jobs that do not fit run direct.  The budget
 * is clamped to the device's free memory less headroom, and if the allocation fails the builds run direct without an error.  J and K
 * are bitwise identical to the direct build.  tuna_set_basis, tuna_set_transform, tuna_set_shard and a new budget drop the store; a
 * stored job whose kept quartet list changes (another tau or density bound) runs direct.  In a group every rank stores its own share.
 * Bases that do not group into shells (per-component kernel) ignore the budget. */
int tuna_set_integral_store(tuna_ctx* ctx, int64_t budget_bytes);
/* info[0] bytes held, [1] work items held, [2] work items of the last build's job set (this rank), [3] builds served by replay. */
int tuna_integral_store_info(const tuna_ctx* ctx, int64_t info[4]);

/* AO -> MO / spin-orbital four-index transformation of a dense ERI tensor (SURVEY.md 8f-2):
 *   tuna_ci.transform_ERI_AO_to_MO(ERI_AO, C, ...)        tuna_ci.py:204-255   so_layout = 0, C1 = C2 = C
 *   tuna_ci.transform_ERI_AO_to_SO(ERI_AO, C_1, C_2, ...)  tuna_ci.py:143-193   so_layout = 1
 * i.e. the einsum chain "mknl,ls->mnks" (C1), "mnks,kr->mnrs" (C2), "mnrs,nq->mqrs" (C1), "mqrs,mp->prqs" (MO) or
 * "mqrs,mp->pqrs" (SO) (C2).  eri is n^4 (NULL = the resident stored tensor, which is left untouched), C1 is n x n1 and
 * C2 is n x n2 (row-major: AO index first).  Output: MO layout [p][r][q][s] = (n2, n2, n1, n1) — interleaved chemists'
 * notation (pr|qs) — or SO layout [p][q][r][s] = (n2, n1, n2, n1).  Four FP64 GEMM-shaped passes on the device. */
int tuna_eri_transform(tuna_ctx* ctx, int n, const double* eri_host, int n1, const double* C1, int n2, const double* C2,
                       int so_layout, double* out_host);
int tuna_eri_transform_dev(tuna_ctx* ctx, int n, const double* d_eri, int n1, const double* dC1, int n2, const double* dC2,
                           int so_layout, double* d_out);
/* The spin-orbital transformation of the post-HF drivers (TUNA/tuna_ci.py:564-570): the reference spin-blocks the AO tensor on the host,
 *   ERI_spin_block = np.kron(np.eye(2), np.kron(np.eye(2), ERI_AO).T)            (16 n^4 doubles)
 * and hands it to transform_ERI_AO_to_SO with spin-blocked coefficients C (2n x n_so).  Here the spin-blocked tensor is formed on the
 * device from the RESIDENT stored tensor (dimension n = the stored dimension) and transformed in place: C1 (2n x n1), C2 (2n x n2),
 * output layout as tuna_eri_transform with so_layout. */
int tuna_eri_transform_spin_blocked(tuna_ctx* ctx, int n1, const double* C1, int n2, const double* C2, int so_layout, double* out_host);

/* One-electron integrals (SURVEY.md 8f-3) of the basis given to tuna_set_basis, in the Cartesian basis:
 *   tuna_integral.calculate_one_electron_integrals(n_basis, basis_functions, n_atoms, atoms, dipole_origin, num_threads)   pyx:282-445
 * S overlap, T kinetic energy, V nuclear attraction (sum over the n_atoms nuclei at atom_z with charges atom_charge, all on the z
 * axis like the reference's own nuclear integral, pyx:783), D[3] dipole (x, y, z) and Q[3] diagonal quadrupole (xx, yy, zz)
 * about dipole_origin[3].  S, T, V: n x n; D, Q: 3 x n x n. */
int tuna_one_electron(tuna_ctx* ctx, int n_atoms, const double* atom_z, const double* atom_charge, const double* dipole_origin,
                      double* S, double* T, double* V, double* D, double* Q);
/* tuna_integral.calculate_cross_basis_overlap_matrix (pyx:626-778): S12[i][j] = <bf_1[i] | bf_2[j]> for two independent bases,
 * each passed like the arguments of tuna_set_basis.  Needs no basis in the context. */
int tuna_cross_overlap(tuna_ctx* ctx, int n1, const double* origins_z1, const int32_t* lmn1, const int32_t* nprim1, const int64_t* prim_offset1,
                       const double* exps1, const double* coef_eff1, int n2, const double* origins_z2, const int32_t* lmn2, const int32_t* nprim2,
                       const int64_t* prim_offset2, const double* exps2, const double* coef_eff2, double* S12);

/* Introspection for tests and bench.py.
 * counts[0] AO pairs, [1] unique AO quartets, [2] quartets passing the x/y parity test (pyx:1324-1327),
 * [3] primitive quartets among those, [4] quartets evaluated by the last direct build (after screening, this rank),
 * [5] kernels launched by this context so far, [6] ncart, [7] nbf. */
int tuna_get_counts(const tuna_ctx* ctx, int64_t counts[8]);
/* Device time (ms, CUDA events on the launching stream) of the dominant kernel of the last call:
 * which = 0 ERI fill, 1 cart->sph, 2 stored J/K, 3 direct J/K (the accumulation of the last density pass), 4 AO->MO transformation,
 * 5 one-electron integrals, 6 on ctxs[0] of a tuna_jk_direct_group call with nctx > 1: from the end of the last rank's accumulation to
 * J/K ready (pull, sum, finish) of the last density pass.  Synchronises the stream. */
int tuna_last_kernel_ms(tuna_ctx* ctx, int which, float* ms);
/* Algorithmic FP64 flop count of the reference algorithm for the parity-surviving unique quartets of the
 * current basis (formula F(a,b) of SURVEY.md section 8d), and the J/K digestion flops per density. */
int tuna_algorithmic_flops(const tuna_ctx* ctx, double* eri_flops, double* digest_flops_per_density);
/* Dependency-free DFMA stream used to measure the FP64 pipe peak of this device (TFLOP/s). */
int tuna_fp64_peak_probe(tuna_ctx* ctx, double* tflops);

#ifdef __cplusplus
}
#endif
#endif
