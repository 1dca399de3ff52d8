// tuna_b200.cu — sm_100a kernels + C ABI (include/tuna_b200.h) of the TUNA SCF two-electron provider.
//
// Kernels (DESIGN.md has the roofline of each):
//   k_fill_scatter    dense tensor, second pass: the engine's fill mode (k_shell4_*) leaves the unique integrals of every work item in
//                     scratch rows; this sums the primitive chunks in a fixed order and writes the eight images
//   k_fill_scatter_sph  the same second pass straight into the spherical tensor: each shell quartet's Cartesian block is rotated with
//                     the per-shell blocks of U and written to the eight images; no Cartesian tensor exists
//   k_eri_fill        the dense tensor with one thread per AO quartet (uncontracted bases, bases that do not group into shells)
//   k_schwarz         Q_ij = sqrt((ij|ij))
//   k_rotate_axis     one index of the Cartesian->spherical rotation (sparse U), used 4x for the tensor, 2x for matrices
//   k_jk_stored_sym / _tma / k_jk_stored   fused single-pass J+K over the resident dense tensor (HBM-bound), atomic-free
//   k_shell4_one / k_shell4_multi          direct J/K: the shell-quartet engine of shell4.cuh (one class job per launch / all light
//                                          class jobs of one group size in one persistent launch), reproducible integer accumulation
//   k_jk_direct       per-component direct J/K for bases that do not group into full shells (FP64 atomics)
//   k_density_scan / k_density_split / k_add_into   device densities of any real P: max|P| and max|P - P^T|, the split into symmetric
//                     and antisymmetric parts, K[S] + K[A]
//   k_axis_gemm, k_spin_block              AO->MO / spin-orbital transformation on the FP64 tensor cores (mo_transform.cuh)
//   k_one_electron, k_cross_overlap        one-electron integrals (oneel_core.cuh)
// Reference being replaced: TUNA/tuna_integrals/tuna_integral.pyx:1267-1355 (ERI driver), TUNA/tuna_kernel.py:504-523
// (rotation), TUNA/tuna_scf.py:27-72 (J/K einsums).  No CPU fallback exists in this file.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include <map>
#include <new>
#include <string>
#include <thread>
#include <vector>

#include "../../include/tuna_b200.h"
#include "density_split.hpp"
#include "devbuf.hpp"
#include "eri_core.cuh"
#include "pairtable.hpp"
#include "shell_host.hpp"
#include "shell_jk.cuh"
#include "shell4_host.hpp"
#include "mo_transform.cuh"
#include "oneel_core.cuh"

using namespace tuna;

// ------------------------------------------------------------------------------------------------
// context
// ------------------------------------------------------------------------------------------------
struct CsrDev {
    int rows = 0, cols = 0;
    DevBuf<int> rowptr, col;
    DevBuf<double> val;
};

struct tuna_ctx {
    int device = 0;
    cudaStream_t own_stream = nullptr, stream = nullptr;
    std::string err;
    int64_t launches = 0;
    int sm_count = 148;

    DevBuf<double> d_boys, d_herm;

    // basis + pair table
    HostBasis hb;
    PairTable pt;
    bool pairs_ready = false;         // the AO-pair table is built on first use by an ERI / J/K call (one-electron integrals do not need it)
    int ncart = 0;
    DevBuf<int> d_pi, d_pj, d_cls, d_npp;
    DevBuf<int64_t> d_ppoff;
    DevBuf<double> d_pp;
    DevBuf<double> d_Q;               // Schwarz factor per sorted pair (lazy)
    int64_t task_begin[5] = {0, 0, 0, 0, 0};
    int64_t n_unique = 0, n_surviving = 0, n_primq = 0, n_eval_last = 0;
    double alg_eri_flops = 0, alg_digest_flops = 0;

    // transform
    int nbf = 0;
    bool U_identity = false;
    CsrDev U, Ut;
    // U is block-diagonal over the engine's shells with one x/y parity per row (build_sph_shells): tuna_eri_fill_sph rotates shell
    // quartet by shell quartet with these per-shell blocks
    bool U_shell_blocks = false;
    DevBuf<int> d_sph_n, d_sph_idx, d_sph_uoff, d_sph_par;
    DevBuf<double> d_sph_u;

    // dense tensors
    DevBuf<double> d_eri_cart;
    DevBuf<double> d_eri_sph;         // "stored" tensor of dimension n_stored
    int n_stored = 0;
    bool eri_pair_sym = false;        // (il|kj) == (kj|il) holds for the stored tensor: the symmetric streaming J/K kernel may be used

    // J/K workspaces
    DevBuf<double> d_P, d_J, d_K;                  // nD * n^2 staging (spherical)
    DevBuf<double> d_Pc, d_Jc, d_Kc, d_tmp;        // Cartesian
    DevBuf<double> d_Kpart;
    DevBuf<double> d_fnorm;           // per-component norms (shell engine fill mode)
    PinnedBuf<double> h_pin;
    DevBuf<unsigned long long> d_scalars;      // [0] max|P| bits, [1] evaluated-quartet counter, [2..3] read back by the caller (k_pair_sym_check, k_density_scan)
    PinnedBuf<unsigned long long> h_scan;      // tuna_jk_direct_general_dev: the two maxima of k_density_scan, read back

    int shard_rank = 0, shard_n = 1;
    cudaEvent_t ev[7][2] = {};
    uint64_t basis_sum = 0, U_sum = 0;     // checksums of the arrays given to tuna_set_basis / tuna_set_transform (tuna_jk_direct_group)

    // AO -> MO four-index transformation (mo_transform.cuh): two ping-pong work buffers, grown on demand
    DevBuf<double> d_mo_ws[2];

    // shell-quartet engine (shell_jk.cuh)
    ShellTab stab;
    ShellSystem ss;
    bool shell_ready = false;
    DevBuf<int> d_pairA, d_pairB; DevBuf<long long> d_pair_rec; DevBuf<double> d_rec, d_pairQ;
    DevBuf<int> d_sh_ao, d_class_lists; DevBuf<double> d_finv;
    DevBuf<double> d_eval;
    std::vector<size_t> class_list_off;
    static constexpr int NAUX = 16;
    int naux = 16;                   // streams in use (TUNA_B200_STREAMS, 1..16; measured: 16 helps the launch-bound small systems, neutral at nbf 800)
    cudaStream_t aux[NAUX] = {};     // class jobs of one build are independent (integer-atomic accumulation): launches are dealt round-robin to these streams
    cudaEvent_t ev_fork = nullptr, ev_join[NAUX] = {};
    // generation-4 shell engine (shell4.cuh): per-class tables and the job list; the pair data above is shared
    struct ClassTab4Dev { Class4Host host; Class4Dev view; DevBuf<unsigned char> blob; };
    struct Job4Host { Shell4Job job; int G = 1, threads = 128, gpc = 1, nb = 1; size_t smem = 0; double allowed = 0; bool own_launch = true;
                      int cb = 0, ck = 0;            // bra / ket pair class
                      uint64_t list_sum = 0;         // checksum of the kept quartet list (item prefix): the integral store's validity key
                      double cost_per_byte = 0;      // estimated phase 0-4 work of a work item over the bytes of its stored row
                      long long unit0 = 0; };        // flat index of the job's first unit in its launch (grouped jobs: the unit prefix)
    std::map<int, ClassTab4Dev> class_tabs4;     // key La | Lb<<4 | Lc<<8 | Ld<<12 | nD<<16
    // job lists are cached per (threshold, densities per pass, rank count): a build with nD = 5 runs passes of 2, 2 and 1 densities, and
    // direct SCF alternates between thresholds rarely - none of that may rebuild lists or reallocate inside a Fock build
    struct Group4 { int G = 1, threads = 128, njobs = 0, job_off = 0, ctas_per_sm = 1; long long nunits = 0; size_t smem = 0;
                    DevBuf<Shell4Job> d_jobs; DevBuf<long long> d_unit_prefix;         // light jobs of one group size in one persistent launch
                    std::vector<int> members; std::vector<Shell4Job> host_jobs; };     // indices into JobSet4::jobs, the descriptors as in d_jobs
    struct JobSet4 { double tau = -1.0, dens_bound = 0.0; int nD = 0, shard_n = 0; std::vector<Job4Host> jobs; std::vector<Group4> groups; DevBuf<long long> d_prefix;
                     // fill job set (nD == 0): scratch rows of all work items, every job's descriptor and the prefix of (shell quartet, fill entry) counts for the scatter pass
                     DevBuf<double> d_scratch; DevBuf<Shell4Job> d_all_jobs; DevBuf<long long> d_scatter_pre; long long scatter_total = 0;
                     DevBuf<int> d_fill_pairs; };
    std::vector<JobSet4> jobsets4;
    int cur_jobset4 = -1;
    // The job lists are pre-screened on the host with tau / dens_bound, dens_bound = an upper bound of max |P| in the engine's working
    // basis; the device applies the exact test Q_ab Q_cd max|P| < tau.  1e3 covers |P| <= ~10 in the spherical basis (the Cartesian
    // back-rotation of an h shell can amplify by ~1e2).  tuna_jk_direct and tuna_jk_direct_general_dev set it from max|P| (plan_density);
    // callers of tuna_jk_direct_dev with larger densities scale them down (J and K are linear in P).
    double dens_bound = 1e3;
    DevBuf<long long> d_fix;          // reproducible accumulation: [J hi | J lo | K hi | K lo], nD * ncart^2 words each
    DevBuf<long long> d_peer;         // tuna_jk_direct_group on ctxs[0]: the other ranks' accumulators, pulled for k_fix_reduce
    cudaEvent_t ev_group = nullptr;                      // tuna_jk_direct_group: cross-device ordering (density ready / accumulate done / pulled)
    unsigned long long peers_tried = 0;                  // tuna_jk_direct_group on ctxs[0]: devices whose peer access with this one was requested
    CsrDev Uf, Uft;                 // U * diag(f) and its transpose: per-component norms folded into the rotation
    int direct_engine = 1;          // 1 = shell engine when the basis groups into shells, 0 = per-component kernel

    // integral store (semi-direct J/K, tuna_set_integral_store): the contracted integral buffers of whole class jobs, one row per work
    // item of this rank, planned at the first direct build after the store was set or dropped and filled by that build
    struct StoreEntry { int cb, ck, psplit, chunk, nint; uint64_t list_sum; long long unit0, base, items; bool filled; };
    int64_t store_budget = 0;        // bytes asked for; 0 = off
    bool store_planned = false;
    std::vector<StoreEntry> store;
    DevBuf<double> d_store;
    int64_t store_replays = 0, store_items_last = 0;
    bool store_served = false;       // a job of the current build ran from the store
};

#define CK(call)                                                                                   \
    do {                                                                                           \
        cudaError_t e_ = (call);                                                                   \
        if (e_ != cudaSuccess) {                                                                   \
            ctx->err = std::string(#call) + ": " + cudaGetErrorString(e_);                         \
            return (e_ == cudaErrorMemoryAllocation) ? TUNA_ERR_NOMEM : TUNA_ERR_CUDA;             \
        }                                                                                          \
    } while (0)

#define FAIL(code, msg) do { ctx->err = (msg); return (code); } while (0)

// At least n elements in buf (DevBuf::grow); on failure ctx->err says why and the caller returns TUNA_ERR_NOMEM.
#define GROW(buf, n) do { if (const int rc_ = (buf).grow((n), ctx->err)) return rc_; } while (0)

// No exception may cross the C ABI (include/tuna_b200.h): every entry point that touches std containers is a function-try-block.
#define TUNA_CATCH                                                                                                     \
    catch (const std::bad_alloc&) { if (ctx) ctx->err = "host allocation failed"; return TUNA_ERR_NOMEM; }             \
    catch (const std::exception& e_) { if (ctx) ctx->err = std::string("internal error: ") + e_.what(); return TUNA_ERR_STATE; } \
    catch (...) { if (ctx) ctx->err = "internal error"; return TUNA_ERR_STATE; }

// FNV-1a over raw bytes: tuna_jk_direct_group compares the basis and transform of its contexts with it
static uint64_t checksum(const void* p, size_t bytes, uint64_t h = 1469598103934665603ull) {
    const unsigned char* c = static_cast<const unsigned char*>(p);
    for (size_t i = 0; i < bytes; ++i) h = (h ^ c[i]) * 1099511628211ull;
    return h;
}

static int check_pair_symmetry(tuna_ctx* ctx);
static int ensure_shell4(tuna_ctx* ctx, double tau, int nD);
static int launch_shell4_jobs(tuna_ctx* ctx, int nD, const double* Pc, const double* Psym, double* Jc, double* Kc, double tau, long long fix_lo);
static void drop_store(tuna_ctx* ctx);


// Opt-in to more than 48 KB of dynamic shared memory.  The attribute is PER DEVICE (a process may hold contexts on several GPUs), so the
// "already done" flag is a bit per device ordinal, one flag word per kernel instantiation.
// tuna_jk_direct_group enqueues from one host thread per device, hence the atomic.
template <auto Kernel>
static cudaError_t opt_in_smem(const tuna_ctx* ctx) {
    static std::atomic<unsigned long long> done{0};
    const unsigned long long bit = 1ull << (ctx->device & 63);
    if (done.load() & bit) return cudaSuccess;
    const cudaError_t e = cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) done.fetch_or(bit);
    return e;
}


// ------------------------------------------------------------------------------------------------
// device helpers
// ------------------------------------------------------------------------------------------------
struct PairTableDev {
    const int* pi; const int* pj; const int* cls; const int* npp; const int64_t* ppoff; const double* pp;
    int64_t gbeg[5];     // pair index range of each parity group
    int64_t tbeg[5];     // task (quartet) index range of each parity group
};

__device__ __forceinline__ PairClass unpack_cls(int c) { return PairClass{c & 255, (c >> 8) & 255, c >> 16}; }

// task index -> (a >= b) sorted pair indices within a parity group
__device__ __forceinline__ void decode_task(const PairTableDev& T, int64_t t, int64_t& a, int64_t& b) {
    int g = 0;
    if (t >= T.tbeg[1]) g = 1;
    if (t >= T.tbeg[2]) g = 2;
    if (t >= T.tbeg[3]) g = 3;
    int64_t u = t - T.tbeg[g];
    int64_t r = (int64_t)((sqrt(8.0 * (double)u + 1.0) - 1.0) * 0.5);
    while (r * (r + 1) / 2 > u) --r;
    while ((r + 1) * (r + 2) / 2 <= u) ++r;
    a = T.gbeg[g] + r;
    b = T.gbeg[g] + (u - r * (r + 1) / 2);
}

__device__ __forceinline__ double quartet_value(const PairTableDev& T, int64_t a, int64_t b, const double* boys, const double* herm) {
    return eri_ao_quartet(T.pp + T.ppoff[a] * PP_DOUBLES, T.npp[a], T.pp + T.ppoff[b] * PP_DOUBLES, T.npp[b],
                          unpack_cls(T.cls[a]), unpack_cls(T.cls[b]), boys, herm);
}

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
// Dense fill: one thread per unique parity-surviving AO quartet; parity-forbidden entries stay zero from the memset.
// Heavily contracted quartets (more than 32 primitive quartets) are shared by the 32 lanes of the warp, so the few
// (ss|ss)-type quartets of a contracted basis no longer serialise thousands of primitive quartets in one thread.
__global__ void __launch_bounds__(128) k_eri_fill(PairTableDev T, const double* __restrict__ boys, const double* __restrict__ herm,
                                                  double* __restrict__ out, int n) {
    const int64_t ntask = T.tbeg[4];
    const int64_t n1 = n, n2 = n1 * n1, n3 = n2 * n1;
    const int lane = threadIdx.x & 31;
    const int64_t warp0 = ((int64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5, nwarps = ((int64_t)gridDim.x * blockDim.x) >> 5;
    for (int64_t base = warp0 * 32; base < ntask; base += nwarps * 32) {
        const int64_t t = base + lane;
        const bool valid = t < ntask;
        int64_t a = 0, b = 0;
        int nq = 0;
        if (valid) {
            decode_task(T, t, a, b);
            nq = T.npp[a] * T.npp[b];
        }
        const bool heavy = nq > 32;
        double v = (valid && !heavy) ? quartet_value(T, a, b, boys, herm) : 0.0;
        unsigned mask = __ballot_sync(0xffffffffu, heavy);
        while (mask) {
            const int src = __ffs(mask) - 1;
            mask &= mask - 1;
            const int64_t as = __shfl_sync(0xffffffffu, a, src), bs = __shfl_sync(0xffffffffu, b, src);
            double part = eri_ao_quartet_strided(T.pp + T.ppoff[as] * PP_DOUBLES, T.npp[as], T.pp + T.ppoff[bs] * PP_DOUBLES, T.npp[bs],
                                                 unpack_cls(T.cls[as]), unpack_cls(T.cls[bs]), boys, herm, lane, 32);
            for (int o = 16; o > 0; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
            if (lane == src) v = part;
        }
        if (valid) {
            const int64_t i = T.pi[a], j = T.pj[a], k = T.pi[b], l = T.pj[b];
            out[i * n3 + j * n2 + k * n1 + l] = v; out[k * n3 + l * n2 + i * n1 + j] = v;
            out[j * n3 + i * n2 + l * n1 + k] = v; out[l * n3 + k * n2 + j * n1 + i] = v;
            out[j * n3 + i * n2 + k * n1 + l] = v; out[l * n3 + k * n2 + i * n1 + j] = v;
            out[i * n3 + j * n2 + l * n1 + k] = v; out[k * n3 + l * n2 + j * n1 + i] = v;
        }
    }
}

__global__ void __launch_bounds__(128) k_schwarz(PairTableDev T, const double* __restrict__ boys, const double* __restrict__ herm,
                                                 double* __restrict__ Q, int64_t npair) {
    for (int64_t a = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; a < npair; a += (int64_t)gridDim.x * blockDim.x)
        Q[a] = sqrt(fabs(quartet_value(T, a, a, boys, herm)));
}

__global__ void k_eri_single(const double* __restrict__ ppA, int nA, int clsA, const double* __restrict__ ppB, int nB, int clsB,
                             const double* __restrict__ boys, const double* __restrict__ herm, double* out) {
    if (threadIdx.x == 0 && blockIdx.x == 0)
        *out = eri_ao_quartet(ppA, nA, ppB, nB, unpack_cls(clsA), unpack_cls(clsB), boys, herm);
}

// out[o, p, r] = sum_e val[e] * in[o, col[e], r] over the CSR row p: one index of a tensor rotated by a sparse matrix.
// Two index mappings without 64-bit divisions in the element loop:
//   k_rotate_axis_wide  (inner >= 128): one (o, p) row per blockIdx.x, threads stride over r -> coalesced loads and stores;
//   k_rotate_axis_narrow (inner < 128): one o per blockIdx.x, threads stride over the contiguous (p, r) block of that o.
__global__ void __launch_bounds__(256) k_rotate_axis_wide(const double* __restrict__ in, double* __restrict__ out, const int* __restrict__ rowptr,
                                                          const int* __restrict__ col, const double* __restrict__ val, int n_in, int n_out,
                                                          int64_t inner) {
    const int64_t op = blockIdx.x;
    const int p = (int)(op % n_out);
    const int64_t o = op / n_out;
    const int e0 = rowptr[p], e1 = rowptr[p + 1];
    const double* src = in + o * n_in * inner;
    double* dst = out + op * inner;
    for (int64_t r = (int64_t)blockIdx.y * blockDim.x + threadIdx.x; r < inner; r += (int64_t)gridDim.y * blockDim.x) {
        double s = 0.0;
        for (int e = e0; e < e1; ++e) s = fma(val[e], src[(int64_t)col[e] * inner + r], s);
        dst[r] = s;
    }
}

__global__ void __launch_bounds__(256) k_rotate_axis_narrow(const double* __restrict__ in, double* __restrict__ out, const int* __restrict__ rowptr,
                                                            const int* __restrict__ col, const double* __restrict__ val, int64_t outer, int n_in,
                                                            int n_out, int inner) {
    const int block_elems = n_out * inner;
    for (int64_t o = blockIdx.x; o < outer; o += gridDim.x) {
        const double* src = in + o * n_in * inner;
        double* dst = out + o * block_elems;
        for (int t = threadIdx.x; t < block_elems; t += blockDim.x) {
            const int p = t / inner, r = t - p * inner;
            double s = 0.0;
            for (int e = rowptr[p]; e < rowptr[p + 1]; ++e) s = fma(val[e], src[col[e] * inner + r], s);
            dst[t] = s;
        }
    }
}


// Fused stored-mode J+K.  Block (chunk c, row i) owns the contiguous slabs E[i, l, :, :], l in the chunk.
// Thread (rt, j): j = tid % n fixed, k = rt, rt + r, ...;  one coalesced read of each element serves
//   J[i,l]  += E[i,l,k,j] * P[k,j]     (block reduction, written once)
//   K[i,j]  += E[i,l,k,j] * P[k,l]     (register accumulator over k and l, written once per block to Kpart)
template <int ND>
__global__ void __launch_bounds__(1024) k_jk_stored(const double* __restrict__ E, const double* __restrict__ P, double* __restrict__ J,
                                                    double* __restrict__ Kpart, int n, int r, int lch, int nchunk) {
    extern __shared__ double sm[];
    const int i = blockIdx.y, c = blockIdx.x;
    const int tid = threadIdx.x, j = tid % n, rt = tid / n;
    const bool active = tid < n * r;                   // blockDim.x is n * r rounded up to a whole warp
    const int nwarp = blockDim.x >> 5, warp = tid >> 5, lane = tid & 31;
    const int l0 = c * lch, l1 = min(n, l0 + lch);
    const size_t nn = (size_t)n * n;
    double* sJ = sm;                                   // [ND][lch][nwarp]
    double* sK = sm + (size_t)ND * lch * nwarp;        // [ND][r][n]
    double accK[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) accK[d] = 0.0;
    for (int l = l0; l < l1; ++l) {
        const double* Eb = E + ((size_t)i * n + l) * nn;
        double accJ[ND];
#pragma unroll
        for (int d = 0; d < ND; ++d) accJ[d] = 0.0;
#pragma unroll 4
        for (int k = active ? rt : n; k < n; k += r) {
            const double e = __ldcs(Eb + (size_t)k * n + j);   // streamed once: evict-first
#pragma unroll
            for (int d = 0; d < ND; ++d) {
                accJ[d] = fma(e, __ldg(P + d * nn + (size_t)k * n + j), accJ[d]);
                accK[d] = fma(e, __ldg(P + d * nn + (size_t)k * n + l), accK[d]);
            }
        }
#pragma unroll
        for (int d = 0; d < ND; ++d) {
            double v = accJ[d];
            for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
            if (lane == 0) sJ[((size_t)d * lch + (l - l0)) * nwarp + warp] = v;
        }
    }
#pragma unroll
    for (int d = 0; d < ND; ++d)
        if (active) sK[((size_t)d * r + rt) * n + j] = accK[d];
    __syncthreads();
    for (int x = tid; x < ND * (l1 - l0); x += blockDim.x) {
        const int d = x / (l1 - l0), ll = x % (l1 - l0);
        double v = 0.0;
        for (int w = 0; w < nwarp; ++w) v += sJ[((size_t)d * lch + ll) * nwarp + w];
        if (J) J[d * nn + (size_t)i * n + l0 + ll] = v;
    }
    if (Kpart)
        for (int x = tid; x < ND * n; x += blockDim.x) {
            const int d = x / n, jj = x % n;
            double v = 0.0;
            for (int q = 0; q < r; ++q) v += sK[((size_t)d * r + q) * n + jj];
            Kpart[(((size_t)d * n + i) * nchunk + c) * n + jj] = v;
        }
}


// ---- stored-mode J/K, TMA-streamed variant ------------------------------------------------------------------------
// The dense tensor is a pure HBM stream (each element is used once per density), so the B200-native shape is a
// persistent CTA per SM that pulls contiguous row tiles of E[i,l,:,:] into a shared-memory ring with 1-D bulk TMA
// copies (cp.async.bulk + mbarrier complete_tx) while the previous tiles are being contracted.  Each CTA owns a
// contiguous range of (i,l) slabs: J[i,l] is written once by its owner, K[i,:] is accumulated in registers and flushed
// to a per-CTA partial row whenever i changes (k_kslot_reduce sums the partial rows in a fixed order) — no atomics.
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void tma_bulk_load(void* dst, const void* src, uint32_t bytes, uint64_t* bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(smem_u32(dst)), "l"(src),
                 "r"(bytes), "r"(smem_u32(bar))
                 : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok = 0;
    while (!ok)
        asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }"
                     : "=r"(ok)
                     : "r"(smem_u32(bar)), "r"(parity)
                     : "memory");
}

constexpr int JK_MAX_STAGES = 4;

template <int ND>
__global__ void __launch_bounds__(1024) k_jk_stored_tma(const double* __restrict__ E, const double* __restrict__ P, double* __restrict__ J,
                                                           double* __restrict__ Kslot, int* __restrict__ Krow, int n, int r, int R, int q,
                                                           int nstage, int kslots) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const size_t tile_doubles = (size_t)R * n;
    double* ring = reinterpret_cast<double*>(smem_raw);
    double* sJ = ring + (size_t)nstage * tile_doubles;                 // [2][nwarp][ND]
    const int nwarp = blockDim.x >> 5, warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    double* sK = sJ + 2 * nwarp * ND;                                   // [ND][r][n]
    uint64_t* bars = reinterpret_cast<uint64_t*>(sK + (size_t)ND * r * n);
    const int tid = threadIdx.x, j = tid % n, rt = tid / n;
    const bool active = tid < n * r;
    const size_t nn = (size_t)n * n;
    // slab range of this CTA (32-bit, incremental indices: no divisions in the tile loop)
    const int total = n * n;
    const int s0 = (int)((long long)total * blockIdx.x / gridDim.x), s1 = (int)((long long)total * (blockIdx.x + 1) / gridDim.x);
    const int ntile = (s1 - s0) * q;
    if (tid == 0) {
        for (int s = 0; s < nstage; ++s) mbar_init(&bars[s], 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    // producer state (thread 0): next tile to issue
    int p_slab = s0, p_part = 0, p_stage = 0, p_issued = 0;
    auto issue = [&]() {
        const int row0 = p_part * R, rows = min(R, n - row0);
        const uint32_t bytes = (uint32_t)(rows * n * (int)sizeof(double));
        mbar_expect_tx(&bars[p_stage], bytes);
        tma_bulk_load(ring + (size_t)p_stage * tile_doubles, E + ((size_t)p_slab * n + row0) * n, bytes, &bars[p_stage]);
        if (++p_part == q) { p_part = 0; ++p_slab; }
        if (++p_stage == nstage) p_stage = 0;
        ++p_issued;
    };
    if (tid == 0)
        while (p_issued < nstage && p_issued < ntile) issue();
    double accK[ND], accJ[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) { accK[d] = 0.0; accJ[d] = 0.0; }
    int cur_i = s0 / n, flushes = 0, jbuf = 0;
    auto flushK = [&]() {
#pragma unroll
        for (int d = 0; d < ND; ++d)
            if (active) sK[((size_t)d * r + rt) * n + j] = accK[d];
        __syncthreads();
        const int slot = blockIdx.x * kslots + flushes;
        for (int x = tid; x < ND * n; x += blockDim.x) {
            const int d = x / n, jj = x % n;
            double v = 0.0;
            for (int qq = 0; qq < r; ++qq) v += sK[((size_t)d * r + qq) * n + jj];
            Kslot[((size_t)slot * ND + d) * n + jj] = v;
        }
        if (tid == 0) Krow[slot] = cur_i;
        __syncthreads();
#pragma unroll
        for (int d = 0; d < ND; ++d) accK[d] = 0.0;
        ++flushes;
    };
    int i = cur_i, l = s0 - cur_i * n, part = 0, st = 0;
    uint32_t parity = 0;
    for (int t = 0; t < ntile; ++t) {
        const int row0 = part * R, rows = min(R, n - row0);
        if (i != cur_i) { flushK(); cur_i = i; }
        mbar_wait(&bars[st], parity);
        const double* tile = ring + (size_t)st * tile_doubles;
        if (active) {
            const double* Pj = P + (size_t)row0 * n + j;       // P[k][j], k = row0 + row
            const double* Pl = P + (size_t)row0 * n + l;       // P[k][l]
#pragma unroll 4
            for (int row = rt; row < rows; row += r) {
                const double e = tile[row * n + j];
#pragma unroll
                for (int d = 0; d < ND; ++d) {
                    accJ[d] = fma(e, __ldg(Pj + d * nn + (size_t)row * n), accJ[d]);
                    accK[d] = fma(e, __ldg(Pl + d * nn + (size_t)row * n), accK[d]);
                }
            }
        }
        const bool slab_done = part == q - 1;
        if (slab_done) {
#pragma unroll
            for (int d = 0; d < ND; ++d) {
                double v = accJ[d];
                for (int o = 16; o > 0; o >>= 1) v += __shfl_down_sync(0xffffffffu, v, o);
                if (lane == 0) sJ[(jbuf * nwarp + warp) * ND + d] = v;
                accJ[d] = 0.0;
            }
        }
        __syncthreads();                         // every thread is done with this stage (and sJ[jbuf] is complete)
        if (tid == 0 && p_issued < ntile) issue();
        if (slab_done) {
            if (warp == 1 % nwarp && lane < ND && J) {        // a warp other than the producer's sums the per-warp partials
                double v = 0.0;
                for (int w = 0; w < nwarp; ++w) v += sJ[(jbuf * nwarp + w) * ND + lane];
                J[lane * nn + (size_t)i * n + l] = v;
            }
            jbuf ^= 1;
        }
        if (++part == q) { part = 0; if (++l == n) { l = 0; ++i; } }
        if (++st == nstage) { st = 0; parity ^= 1; }
    }
    if (ntile > 0) flushK();
}

// K[d][i][j] = sum of the partial rows of the CTAs whose slab range touches row i, in CTA order (deterministic, atomic-free).
// CTA c owns slabs [total*c/G, total*(c+1)/G); its flush number for row i is i - first_row(c).
__global__ void k_kslot_reduce(const double* __restrict__ Kslot, const int* __restrict__ Krow, double* __restrict__ K, int nD, int n, int grid, int kslots) {
    const int64_t total = (int64_t)nD * n * n;
    const long long slabs = (long long)n * n;
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
        const int jj = (int)(x % n), i = (int)((x / n) % n), d = (int)(x / ((int64_t)n * n));
        // CTAs c with [s0(c), s1(c)) intersecting [i n, (i+1) n)
        int c_lo = (int)(((long long)i * n * grid) / slabs);
        while (c_lo > 0 && slabs * c_lo / grid > (long long)i * n) --c_lo;
        double v = 0.0;
        for (int c = c_lo; c < grid; ++c) {
            const long long s0 = slabs * c / grid, s1 = slabs * (c + 1) / grid;
            if (s0 >= (long long)(i + 1) * n) break;
            if (s1 <= (long long)i * n || s1 == s0) continue;
            const int slot = c * kslots + (i - (int)(s0 / n));
            if (Krow[slot] == i) v += Kslot[((size_t)slot * nD + d) * n + jj];
        }
        K[x] = v;
    }
}

// ---- stored J/K, pair-symmetric streaming kernel ------------------------------------------------------------------
// For a tensor with (il|kj) = (kj|il) (every physical ERI tensor; verified on upload) the Coulomb matrix can be accumulated
// WITHOUT a per-slab block reduction:  J[k][j] = sum_{i,l} E[i,l,k,j] P[i,l]  — thread (k, j) keeps J[k][j] in a register
// and multiplies the slab E[i,l,:,:] it streams by the slab-uniform scalar P[i,l].  K[i][j] = sum_{k,l} E[i,l,k,j] P[k,l] is a
// per-thread register as well (summed over the r thread rows when i changes).  The kernel is then a pure TMA stream:
//   * one producer thread issues 1-D bulk copies (cp.async.bulk + mbarrier complete_tx) of 2*T-element tiles into a deep ring
//     (up to 16 stages, ~160 KB in flight per SM) and only waits on per-stage "empty" mbarriers;
//   * the consumer warps never meet at a CTA barrier inside the stream: they wait on the stage's "full" mbarrier, do two
//     FMAs per element and one elected lane per warp arrives on the "empty" mbarrier;
//   * P^T lives in shared memory (P[k][l] for the thread's rows k is a broadcast read).
// Every CTA writes its partial J (registers -> Jpart[cta]) and partial K rows (Kslot); k_sym_reduce sums both in a fixed order.
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

template <int ND, int MT>
__global__ void __launch_bounds__(1024, 1) k_jk_stored_sym(const double* __restrict__ E, const double* __restrict__ P, double* __restrict__ Jpart,
                                                             double* __restrict__ Kslot, int* __restrict__ Krow, int n, int r, int nstage,
                                                             int kslots, int ncons) {
    extern __shared__ __align__(128) unsigned char smem_raw[];
    const int T = r * n, nn = n * n, tileD = 2 * T;
    double* ring = reinterpret_cast<double*>(smem_raw);
    double* Pt = ring + (size_t)nstage * tileD;                 // [ND][l][k] = P[d][k][l]
    double* sK = Pt + (size_t)ND * nn;                           // [2][ND][r][n]
    uint64_t* full = reinterpret_cast<uint64_t*>(sK + (size_t)2 * ND * r * n);
    uint64_t* empty = full + nstage;
    const int tid = threadIdx.x, lane = tid & 31;
    const int s0 = (int)((long long)nn * blockIdx.x / gridDim.x), s1 = (int)((long long)nn * (blockIdx.x + 1) / gridDim.x);
    const int qreal = (nn + tileD - 1) / tileD;                  // tiles per slab (<= MT / 2)
    if (tid == 0) {
        for (int s = 0; s < nstage; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], ncons >> 5); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    for (int x = tid; x < kslots; x += blockDim.x) Krow[blockIdx.x * kslots + x] = -1;
    __syncthreads();
    asm volatile("griddepcontrol.launch_dependents;");          // let the reduction kernel's launch overlap this grid (it waits for our completion)
    if (tid >= ncons) {                                          // producer warp: one thread streams the CTA's slab range
        if (tid == ncons) {
            int st = 0;
            uint32_t ph = 1;                                     // a fresh "empty" barrier passes a wait on the preceding phase
            for (int s = s0; s < s1; ++s)
                for (int p = 0; p < qreal; ++p) {
                    mbar_wait(&empty[st], ph);
                    const int cnt = min(tileD, nn - p * tileD);
                    const uint32_t bytes = (uint32_t)cnt * (uint32_t)sizeof(double);
                    mbar_expect_tx(&full[st], bytes);
                    tma_bulk_load(ring + (size_t)st * tileD, E + (size_t)s * nn + (size_t)p * tileD, bytes, &full[st]);
                    if (++st == nstage) { st = 0; ph ^= 1; }
                }
        }
        return;
    }
    // ---- consumers ----
    for (int x = tid; x < ND * nn; x += ncons) {
        const int d = x / nn, rem = x - d * nn, k = rem / n, l = rem - k * n;
        Pt[(size_t)d * nn + l * n + k] = P[x];
    }
    asm volatile("bar.sync 1, %0;" ::"r"(ncons) : "memory");
    const bool act = tid < T;
    const int j = tid % n, rt = tid / n;
    double accJ[ND][MT], accK[ND];
#pragma unroll
    for (int d = 0; d < ND; ++d) {
        accK[d] = 0.0;
#pragma unroll
        for (int m = 0; m < MT; ++m) accJ[d][m] = 0.0;
    }
    int st = 0, flushes = 0, kb = 0;
    uint32_t ph = 0;
    int cur_i = s0 / n, i = cur_i, l = s0 - cur_i * n;
    auto flushK = [&]() {
        double* buf = sK + (size_t)kb * ND * r * n;
        if (act) {
#pragma unroll
            for (int d = 0; d < ND; ++d) buf[((size_t)d * r + rt) * n + j] = accK[d];
        }
        asm volatile("bar.sync 1, %0;" ::"r"(ncons) : "memory");
        const int slot = blockIdx.x * kslots + flushes;
        for (int x = tid; x < ND * n; x += ncons) {
            const int d = x / n, jj = x - d * n;
            double v = 0.0;
            for (int qq = 0; qq < r; ++qq) v += buf[((size_t)d * r + qq) * n + jj];
            Kslot[((size_t)slot * ND + d) * n + jj] = v;
        }
        if (tid == 0) Krow[slot] = cur_i;
#pragma unroll
        for (int d = 0; d < ND; ++d) accK[d] = 0.0;
        ++flushes;
        kb ^= 1;
    };
    for (int s = s0; s < s1; ++s) {
        if (i != cur_i) { flushK(); cur_i = i; }
        const double* ptl = Pt + (size_t)l * n;
        double pil[ND];
#pragma unroll
        for (int d = 0; d < ND; ++d) pil[d] = ptl[(size_t)d * nn + i];
#pragma unroll
        for (int p = 0; p < MT / 2; ++p) {
            if (p < qreal) {
                mbar_wait(&full[st], ph);
                const double* tile = ring + (size_t)st * tileD;
#pragma unroll
                for (int mm = 0; mm < 2; ++mm) {
                    const int m = 2 * p + mm, k = rt + m * r;
                    if (act && k < n) {
                        const double e = tile[tid + mm * T];
#pragma unroll
                        for (int d = 0; d < ND; ++d) {
                            accJ[d][m] = fma(e, pil[d], accJ[d][m]);
                            accK[d] = fma(e, ptl[(size_t)d * nn + k], accK[d]);
                        }
                    }
                }
                __syncwarp();
                if (lane == 0) mbar_arrive(&empty[st]);
                if (++st == nstage) { st = 0; ph ^= 1; }
            }
        }
        if (++l == n) { l = 0; ++i; }
    }
    if (s1 > s0) flushK();
    if (act) {
#pragma unroll
        for (int d = 0; d < ND; ++d)
#pragma unroll
            for (int m = 0; m < MT; ++m)
                if (rt + m * r < n) Jpart[((size_t)blockIdx.x * ND + d) * nn + tid + m * T] = accJ[d][m];
    }
}

// J[d][e] = sum over CTAs of Jpart, K as in k_kslot_reduce.  A warp owns four consecutive elements: lane = 4 g + ei sums the
// partials of CTAs c = g (mod 8) for element ei (32-byte sectors fully used), then a fixed shuffle tree adds the eight
// groups -> deterministic, and the ~grid/8 loads per lane are independent.
__global__ void __launch_bounds__(256) k_sym_reduce(const double* __restrict__ Jpart, double* __restrict__ J, const double* __restrict__ Kslot,
                                                    const int* __restrict__ Krow, double* __restrict__ K, int nD, int n, int grid, int kslots) {
    asm volatile("griddepcontrol.wait;" ::: "memory");      // programmatic dependent launch: the streaming kernel's results are visible after this
    const int64_t nn = (int64_t)n * n, total = nD * nn;
    const int64_t gx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    const int lane = threadIdx.x & 31, ei = lane & 3, g = lane >> 2;
    const int64_t x = (gx >> 5) * 4 + ei;
    const bool valid = x < total;
    const int64_t d = valid ? x / nn : 0, e = valid ? x % nn : 0;
    double v0 = 0.0, v1 = 0.0;
    if (valid && J) {
        const double* src = Jpart + (size_t)d * nn + e;
        const size_t stride = (size_t)nD * nn;
        for (int c = g; c < grid; c += 16) {
            v0 += src[(size_t)c * stride];
            if (c + 8 < grid) v1 += src[(size_t)(c + 8) * stride];
        }
    }
    double v = v0 + v1;
    v += __shfl_xor_sync(0xffffffffu, v, 4);
    v += __shfl_xor_sync(0xffffffffu, v, 8);
    v += __shfl_xor_sync(0xffffffffu, v, 16);
    if (valid && g == 0 && J) J[x] = v;
    if (valid && g == 1 && K) {
        const long long slabs = nn;
        const int jj = (int)(e % n), i = (int)(e / n);
        int c_lo = (int)(((long long)i * n * grid) / slabs);
        while (c_lo > 0 && slabs * c_lo / grid > (long long)i * n) --c_lo;
        double kv = 0.0;
        for (int c = c_lo; c < grid; ++c) {
            const long long s0 = slabs * c / grid, s1 = slabs * (c + 1) / grid;
            if (s0 >= (long long)(i + 1) * n) break;
            if (s1 <= (long long)i * n || s1 == s0) continue;
            const int slot = c * kslots + (i - (int)(s0 / n));
            if (Krow[slot] == i) kv += Kslot[((size_t)slot * nD + d) * n + jj];
        }
        K[x] = kv;
    }
}

// max |E[i,l,k,j] - E[k,j,i,l]| and max |E| (bit patterns of non-negative doubles order like integers)
__global__ void k_pair_sym_check(const double* __restrict__ E, int n, unsigned long long* out) {
    const int64_t nn = (int64_t)n * n, total = nn * nn;
    double md = 0.0, mx = 0.0;
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
        const int64_t a = x / nn, b = x % nn;
        if (b > a) continue;
        const double u = E[x], w = E[b * nn + a];
        md = fmax(md, fabs(u - w));
        mx = fmax(mx, fmax(fabs(u), fabs(w)));
    }
    for (int o = 16; o > 0; o >>= 1) { md = fmax(md, __shfl_down_sync(0xffffffffu, md, o)); mx = fmax(mx, __shfl_down_sync(0xffffffffu, mx, o)); }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(out, (unsigned long long)__double_as_longlong(md));
        atomicMax(out + 1, (unsigned long long)__double_as_longlong(mx));
    }
}

__global__ void k_kpart_reduce(const double* __restrict__ Kpart, double* __restrict__ K, int nD, int n, int nchunk) {
    const int64_t total = (int64_t)nD * n * n;
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
        const int jj = (int)(x % n);
        const int64_t di = x / n;
        double v = 0.0;
        for (int c = 0; c < nchunk; ++c) v += Kpart[(di * nchunk + c) * n + jj];
        K[x] = v;
    }
}

__global__ void k_absmax(const double* __restrict__ x, int64_t count, unsigned long long* out) {
    double m = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) m = fmax(m, fabs(x[i]));
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

// out = acc + sign * acc^T  (J = Jacc + Jacc^T, K = Kacc + Kacc^T; see k_jk_direct)
__global__ void k_add_transpose(const double* __restrict__ acc, double* __restrict__ out, int nD, int n) {
    const int64_t nn = (int64_t)n * n, total = nD * nn;
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
        const int64_t d = x / nn, ij = x % nn;
        const int i = (int)(ij / n), j = (int)(ij % n);
        out[x] = acc[x] + acc[d * nn + (int64_t)j * n + i];
    }
}

// Direct J/K: one thread per unique parity-surviving AO quartet (a >= b in the sorted pair order), Schwarz-screened.
// Symmetric P.  With v' = v * (1/2 if i==j) * (1/2 if k==l) * (1/2 if a==b), the 8 images of (ij|kl) reduce to
//   Jacc[i,j] += v' (P[k,l] + P[l,k])      Jacc[k,l] += v' (P[i,j] + P[j,i])
//   Kacc[i,l] += v' P[k,j]   Kacc[j,l] += v' P[k,i]   Kacc[i,k] += v' P[l,j]   Kacc[j,k] += v' P[l,i]
// followed by J = Jacc + Jacc^T, K = Kacc + Kacc^T (k_add_transpose).
__global__ void __launch_bounds__(128) k_jk_direct(PairTableDev T, const double* __restrict__ boys, const double* __restrict__ herm,
                                                   const double* __restrict__ Q, const double* __restrict__ P, double* __restrict__ Jacc,
                                                   double* __restrict__ Kacc, int n, int nD, double tau,
                                                   const unsigned long long* scalars_in, unsigned long long* counter,
                                                   int rank, int nranks) {
    const int64_t ntask = T.tbeg[4];
    const int64_t nn = (int64_t)n * n;
    const double dmax = __longlong_as_double((long long)scalars_in[0]);
    const double thr = (tau > 0.0 && dmax > 0.0) ? tau / dmax : 0.0;
    constexpr int64_t CHUNK = 1024;
    const int64_t nchunks = (ntask + CHUNK - 1) / CHUNK;
    unsigned long long evaluated = 0;
    for (int64_t ch = (int64_t)blockIdx.x * nranks + rank; ch < nchunks; ch += (int64_t)gridDim.x * nranks) {
        const int64_t tend = min(ntask, (ch + 1) * CHUNK);
        for (int64_t t = ch * CHUNK + threadIdx.x; t < tend; t += blockDim.x) {
            int64_t a, b;
            decode_task(T, t, a, b);
            if (Q[a] * Q[b] < thr) continue;
            ++evaluated;
            double v = quartet_value(T, a, b, boys, herm);
            const int i = T.pi[a], j = T.pj[a], k = T.pi[b], l = T.pj[b];
            if (i == j) v *= 0.5;
            if (k == l) v *= 0.5;
            if (a == b) v *= 0.5;
            for (int d = 0; d < nD; ++d) {
                const double* Pd = P + d * nn;
                double* Jd = Jacc + d * nn;
                double* Kd = Kacc + d * nn;
                atomicAdd(Jd + (int64_t)i * n + j, v * (Pd[(int64_t)k * n + l] + Pd[(int64_t)l * n + k]));
                atomicAdd(Jd + (int64_t)k * n + l, v * (Pd[(int64_t)i * n + j] + Pd[(int64_t)j * n + i]));
                atomicAdd(Kd + (int64_t)i * n + l, v * Pd[(int64_t)k * n + j]);
                atomicAdd(Kd + (int64_t)j * n + l, v * Pd[(int64_t)k * n + i]);
                atomicAdd(Kd + (int64_t)i * n + k, v * Pd[(int64_t)l * n + j]);
                atomicAdd(Kd + (int64_t)j * n + k, v * Pd[(int64_t)l * n + i]);
            }
        }
    }
    for (int o = 16; o > 0; o >>= 1) evaluated += __shfl_down_sync(0xffffffffu, evaluated, o);
    if ((threadIdx.x & 31) == 0 && evaluated) atomicAdd(counter, evaluated);
}

// FP64 pipe peak probe: 8 independent DFMA chains per thread.
__global__ void __launch_bounds__(256) k_dfma_probe(double* out, int iters, double x) {
    double a0 = threadIdx.x, a1 = a0 + 1, a2 = a0 + 2, a3 = a0 + 3, a4 = a0 + 4, a5 = a0 + 5, a6 = a0 + 6, a7 = a0 + 7;
    const double y = 1.0 - x;
    for (int i = 0; i < iters; ++i) {
        a0 = fma(a0, x, y); a1 = fma(a1, x, y); a2 = fma(a2, x, y); a3 = fma(a3, x, y);
        a4 = fma(a4, x, y); a5 = fma(a5, x, y); a6 = fma(a6, x, y); a7 = fma(a7, x, y);
    }
    const double s = a0 + a1 + a2 + a3 + a4 + a5 + a6 + a7;
    if (s == 123.456) out[0] = s;
}

// ---- shell-quartet engine (shell4.cuh) ------------------------------------------------------------------------------------
template <int GG>
struct DevPolicy {
    static constexpr int G = GG;
    __device__ __forceinline__ static int lane() { return threadIdx.x & (GG - 1); }
    __device__ __forceinline__ static void sync() {
        if constexpr (GG > 32) __syncthreads();
        else if constexpr (GG == 32) __syncwarp();
        else __syncwarp(((1u << GG) - 1u) << ((threadIdx.x & 31) & ~(GG - 1)));     // only the lanes of this group
    }
    __device__ __forceinline__ static void sync_cta() { __syncthreads(); }
    __device__ __forceinline__ static int cta_thread() { return threadIdx.x; }
    __device__ __forceinline__ static int cta_threads() { return blockDim.x; }
    // fill mode and integral store: index of the work item header hq points to (the unit's first work item is kept behind the headers,
    // see shell4_unit)
    __device__ __forceinline__ static long long work_item_of(const Shell4Job& J, const Quartet4* hq) {
        extern __shared__ double smem_all[];
        const Quartet4* hdr0 = reinterpret_cast<const Quartet4*>(smem_all + J.hdr_off);
        return *reinterpret_cast<const long long*>(reinterpret_cast<const char*>(hdr0 + J.chunk) + 8) + (hq - hdr0);
    }
    // M[idx] += v as the order-independent two-word integer accumulation of fixed_split (no floating-point atomics in the engine)
    __device__ __forceinline__ static void accumulate(double* M, int idx, double v, long long fix_lo) {
        long long h, l;
        fixed_split(v, h, l);
        unsigned long long* W = reinterpret_cast<unsigned long long*>(M);
        if (h != 0) atomicAdd(W + idx, (unsigned long long)h);
        if (l != 0) atomicAdd(W + fix_lo + idx, (unsigned long long)l);
    }
};

// ---- generation-4 engine: one class job per launch, the descriptor travels as a kernel parameter ------------------------------
// A CTA work unit (= multi-GPU sharding unit) is J.chunk consecutive shell quartets; the unit's quartets are decoded ONCE (item ->
// bra / ket pair, Schwarz test, degeneracy weight) into shared-memory headers, then the CTA's groups take them NB at a time.
// Register budget of the engine kernels.  Measured on the B200 (profiles/r02u_register_budget.log): 64 -> 1297 ms per ET800 build (208 B of
// spills in the two-quartet instantiations), 72 -> 1254, 80 -> 1205, 88 -> 1231, 96 -> 1231: 80 registers remove the spills at 3/4 of the
// thread occupancy, which the latency-bound phases tolerate.
#ifndef TUNA_SHELL4_REGS
#define TUNA_SHELL4_REGS 80
#endif
// One CTA work unit: decode the unit's work items ONCE (item -> bra / ket pair, Schwarz test, degeneracy weight, record offsets) into the
// shared-memory headers, then let the CTA's groups take them NB at a time.  SEMI: see shell4_quartets.
template <int GG, int NB, bool SEMI>
__device__ __forceinline__ void shell4_unit(const Shell4Job& J, const ShellData& D, long long unit, int nD, const double* __restrict__ Pf,
                                            const double* __restrict__ Psym, double* Jf, double* Kf, int ncart, double tau, double dmax,
                                            double* smem_all, int& tab_chunk, double& done) {
    const int gpc = blockDim.x / GG, gid = threadIdx.x / GG;
    unsigned* tab = reinterpret_cast<unsigned*>(smem_all + J.tab_off);
    Quartet4* hdr = reinterpret_cast<Quartet4*>(smem_all + J.hdr_off);
    const int CH = J.chunk;
    int& s_ib0 = *reinterpret_cast<int*>(hdr + CH);
    double* sm = smem_all + (size_t)gid * NB * J.total;
    const long long nwi = J.nitems * J.psplit;          // work items: (shell quartet, chunk of bra primitive pairs)
    const long long first = unit * CH;
    __syncthreads();                                  // the previous unit's headers are no longer needed (and the tables are in place)
    if (threadIdx.x == 0) {
        const long long first_item = first / J.psplit;
        int lo = 0, hi = J.nbra;                      // invariant: prefix[lo] <= first_item < prefix[hi]
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (J.item_prefix[mid] <= first_item) lo = mid; else hi = mid;
        }
        s_ib0 = lo;
        *reinterpret_cast<long long*>(reinterpret_cast<char*>(hdr + CH) + 8) = first;      // read by DevPolicy::work_item_of (fill mode, integral store)
    }
    __syncthreads();
    for (int k = threadIdx.x; k < CH; k += blockDim.x) {
        const long long wi = first + k, item = wi / J.psplit;
        const int pchunk = (int)(wi - item * J.psplit);
        Quartet4 h;
        h.active = 0; h.shA = h.shB = h.shC = h.shD = 0; h.ia0 = 0; h.w = 0.0; h.recA = h.recC = 0; h.pA = h.pC = 1.0; h.zA = h.zC = 0.0;
        if (wi < nwi) {
            int ib = s_ib0;
            { const int bchunk = pchunk / J.ksplit; h.ia0 = bchunk * J.clen | ((pchunk - bchunk * J.ksplit) * J.klen) << 16; }
            while (J.item_prefix[ib + 1] <= item) ++ib;
            const int pab = J.bra_list[ib], pcd = J.ket_list[(int)(item - J.item_prefix[ib])];
            h.active = !(tau > 0.0 && D.pairQ[pab] * D.pairQ[pcd] * dmax < tau);
            if (SEMI && !h.active && J.store_mode == S4_STORE) h.active = S4_ONLY_STORE;      // stored for later builds, not digested in this one
            h.shA = D.pairA[pab]; h.shB = D.pairB[pab]; h.shC = D.pairA[pcd]; h.shD = D.pairB[pcd];
            const bool ab = h.shA == h.shB, cd = h.shC == h.shD, dg = pab == pcd;
            h.w = J.fill_scratch ? 1.0 : (ab ? 0.5 : 1.0) * (cd ? 0.5 : 1.0) * (dg ? 0.5 : 1.0);      // fill mode stores plain integrals
            h.recA = D.pair_rec[pab]; h.recC = D.pair_rec[pcd];
            if (h.active) {
                h.pA = D.rec[h.recA]; h.zA = D.rec[h.recA + 1]; h.pC = D.rec[h.recC]; h.zC = D.rec[h.recC + 1];
                if (pchunk == 0 && (!SEMI || h.active == 1)) done += J.uniq[dg ? (ab ? 5 : 4) : (ab ? (cd ? 3 : 1) : (cd ? 2 : 0))];
            }
        }
        hdr[k] = h;
    }
    __syncthreads();
    for (int k0 = 0; k0 < CH; k0 += gpc * NB)
        shell4_quartets<DevPolicy<GG>, NB, SEMI>(J, D, hdr + k0 + gid * NB, sm, tab, tab_chunk, nD, Pf, Psym, Jf, Kf, ncart);
}

// Heavy class jobs: one job per launch, the descriptor travels as a kernel parameter (constant bank / uniform registers).  A CTA work
// unit (= multi-GPU sharding unit) is J.chunk consecutive work items.
template <int GG, int NB, int REGS = TUNA_SHELL4_REGS, bool SEMI = false>
__global__ void __launch_bounds__((GG > 128) ? GG : 128, 65536 / (((GG > 128) ? GG : 128) * REGS))
k_shell4_one(Shell4Job J, ShellData D, int nD, const double* __restrict__ Pf, const double* __restrict__ Psym, double* Jf, double* Kf, int ncart,
             double tau, const unsigned long long* scalars, double* evaluated, int rank, int nranks) {
    extern __shared__ double smem_all[];
    const double dmax = __longlong_as_double((long long)scalars[0]);
    const long long nunit = (J.nitems * J.psplit + J.chunk - 1) / J.chunk;
    shell4_load_tables<NB>(J.ct, 0, reinterpret_cast<unsigned*>(smem_all + J.tab_off), threadIdx.x, blockDim.x, J.oIt, J.oP);
    int tab_chunk = 0;
    double done = 0.0;
    for (long long gc = (long long)blockIdx.x * nranks + rank; gc < nunit; gc += (long long)gridDim.x * nranks)
        shell4_unit<GG, NB, SEMI>(J, D, gc, nD, Pf, Psym, Jf, Kf, ncart, tau, dmax, smem_all, tab_chunk, done);
    if (done != 0.0) atomicAdd(reinterpret_cast<unsigned long long*>(evaluated), (unsigned long long)(done + 0.5));      // integer counter: no FP64 atomics in the engine
}

// Light class jobs: ALL jobs of one launch geometry (group size, quartets per batch) in ONE persistent launch.  Small systems are bound by
// the launch count (N2/cc-pVTZ: 231 class jobs of ~10 us each).  The work units of the jobs form one flat list (unit_prefix); a CTA walks
// it with a grid stride (dealt round-robin to ranks like the single-job kernel) and keeps the descriptor of its current job in shared
// memory, reloading descriptor and digestion tables when it crosses into the next job.
template <int GG, int NB, bool SEMI = false>
__global__ void __launch_bounds__((GG > 128) ? GG : 128, 65536 / (((GG > 128) ? GG : 128) * TUNA_SHELL4_REGS))
k_shell4_multi(const Shell4Job* __restrict__ jobs, const long long* __restrict__ unit_prefix, int njobs, int job_off, ShellData D, int nD,
               const double* __restrict__ Pf, const double* __restrict__ Psym, double* Jf, double* Kf, int ncart, double tau,
               const unsigned long long* scalars, double* evaluated, int rank, int nranks) {
    extern __shared__ double smem_all[];
    Shell4Job& J = *reinterpret_cast<Shell4Job*>(smem_all + job_off);          // behind the largest job's areas
    const double dmax = __longlong_as_double((long long)scalars[0]);
    const long long nunits = unit_prefix[njobs];
    int cur = -1, tab_chunk = -1;
    double done = 0.0;
    for (long long u = (long long)blockIdx.x * nranks + rank; u < nunits; u += (long long)gridDim.x * nranks) {
        int lo = 0, hi = njobs;                         // job of this unit (uniform in the CTA)
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (unit_prefix[mid] <= u) lo = mid; else hi = mid;
        }
        if (lo != cur) {
            __syncthreads();                            // everybody is done with the previous job's descriptor and tables
            const int* src = reinterpret_cast<const int*>(jobs + lo);
            int* dst = reinterpret_cast<int*>(&J);
            for (int x = threadIdx.x; x < (int)(sizeof(Shell4Job) / sizeof(int)); x += blockDim.x) dst[x] = src[x];
            __syncthreads();
            shell4_load_tables<NB>(J.ct, 0, reinterpret_cast<unsigned*>(smem_all + J.tab_off), threadIdx.x, blockDim.x, J.oIt, J.oP);
            cur = lo; tab_chunk = 0;
        }
        shell4_unit<GG, NB, SEMI>(J, D, u - unit_prefix[lo], nD, Pf, Psym, Jf, Kf, ncart, tau, dmax, smem_all, tab_chunk, done);
    }
    if (done != 0.0) atomicAdd(reinterpret_cast<unsigned long long*>(evaluated), (unsigned long long)(done + 0.5));      // integer counter: no FP64 atomics in the engine
}

// Dense fill, second pass (shell4_fill_scatter).  A block takes a group of whole shell quartets of one class job (256 / nfill of them, at
// least one) and runs the four scatter modes over the group back to back, so the scratch rows come from DRAM once (the permuted re-reads
// of modes 1-3 hit L2) and the lanes of every mode write runs of consecutive tensor elements.  group_pre = prefix of groups per job.
__global__ void __launch_bounds__(256) k_fill_scatter(const Shell4Job* __restrict__ jobs, const long long* __restrict__ group_pre, int njobs, ShellData D,
                                                      const double* __restrict__ fnorm, double* __restrict__ out, int n) {
    const long long ngroups = group_pre[njobs];
    for (long long t = blockIdx.x; t < ngroups; t += gridDim.x) {
        int lo = 0, hi = njobs;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (group_pre[mid] <= t) lo = mid; else hi = mid;
        }
        const Shell4Job& J = jobs[lo];
        const int nf = J.ct.nfill, ipg = nf >= 256 ? 1 : 256 / nf;
        const long long item0 = (t - group_pre[lo]) * ipg;
        const int cnt = (int)min((long long)ipg, J.nitems - item0) * nf;
#pragma unroll 1
        for (int mode = 0; mode < 4; ++mode)
            for (int x = threadIdx.x; x < cnt; x += 256) {
                const int k = x / nf;
                shell4_fill_scatter(J, D, item0 + k, x - k * nf, mode, fnorm, out, n);
            }
    }
}

// Spherical fill, second pass (shell4_fill_sph).  Same groups of whole shell quartets as k_fill_scatter; the CTA takes the quartets of a
// group one after another.  Each CTA keeps the Cartesian block of its current quartet in its own slice of `ws` (ws_stride doubles, L2
// resident) and the two contraction buffers (xsize doubles each) in dynamic shared memory.
__global__ void __launch_bounds__(256) k_fill_scatter_sph(const Shell4Job* __restrict__ jobs, const long long* __restrict__ group_pre, int njobs, ShellData D,
                                                          SphData Y, const double* __restrict__ fnorm, double* __restrict__ ws, long long ws_stride,
                                                          int xsize, double* __restrict__ out, int n) {
    extern __shared__ double smem_all[];
    double* cart = ws + blockIdx.x * ws_stride;
    const long long ngroups = group_pre[njobs];
    for (long long t = blockIdx.x; t < ngroups; t += gridDim.x) {
        int lo = 0, hi = njobs;
        while (hi - lo > 1) {
            const int mid = (lo + hi) >> 1;
            if (group_pre[mid] <= t) lo = mid; else hi = mid;
        }
        const Shell4Job& J = jobs[lo];
        const int nf = J.ct.nfill, ipg = nf >= 256 ? 1 : 256 / nf;
        const long long item0 = (t - group_pre[lo]) * ipg, cnt = min((long long)ipg, J.nitems - item0);
#pragma unroll 1
        for (long long k = 0; k < cnt; ++k) shell4_fill_sph<DevPolicy<256>>(J, D, Y, item0 + k, fnorm, cart, smem_all, smem_all + xsize, out, n);
    }
}

// reproducible accumulation: (hi, lo) integer words -> FP64 (fixed_value), J and K in one launch
__global__ void k_fixed_to_double(const long long* __restrict__ fix, double* __restrict__ J, double* __restrict__ K, size_t count) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
        J[i] = fixed_value(fix[i], fix[count + i]);
        K[i] = fixed_value(fix[2 * count + i], fix[3 * count + i]);
    }
}

__global__ void k_absmax_scaled(const double* __restrict__ x, const double* __restrict__ finv, int n, int nD, unsigned long long* out) {
    const int64_t nn = (int64_t)n * n, count = nn * nD;
    double m = 0.0;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (int64_t)gridDim.x * blockDim.x) {
        const int64_t ij = i % nn;
        m = fmax(m, fabs(x[i] * finv[ij / n] * finv[ij % n]));
    }
    for (int o = 16; o > 0; o >>= 1) m = fmax(m, __shfl_down_sync(0xffffffffu, m, o));
    if ((threadIdx.x & 31) == 0) atomicMax(out, (unsigned long long)__double_as_longlong(m));
}

// out = acc + sign_d * acc^T, sign from the bit mask (bit d set -> antisymmetric density d)
__global__ void k_add_transpose_signed(const double* __restrict__ acc, double* __restrict__ out, int nD, int n, unsigned anti_mask) {
    const int64_t nn = (int64_t)n * n, total = nD * nn;
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
        const int64_t d = x / nn, ij = x % nn;
        const int i = (int)(ij / n), j = (int)(ij % n);
        const double t = acc[d * nn + (int64_t)j * n + i];
        out[x] = ((anti_mask >> d) & 1u) ? acc[x] - t : acc[x] + t;
    }
}

// max|P| into out[0] and max|P - P^T| into out[1] over a stack of nD n x n densities (bit patterns of non-negative doubles order like
// integers).  density_extrema takes the same two maxima on the host.
__global__ void k_density_scan(const double* __restrict__ P, int nD, int n, unsigned long long* out) {
    const int64_t nn = (int64_t)n * n, total = nD * nn;
    double pm = 0.0, am = 0.0;
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
        const int64_t d = x / nn, ij = x % nn;
        const int i = (int)(ij / n), j = (int)(ij % n);
        const double v = P[x], t = P[d * nn + (int64_t)j * n + i];
        pm = fmax(pm, fabs(v));
        am = fmax(am, fabs(v - t));
    }
    for (int o = 16; o > 0; o >>= 1) { pm = fmax(pm, __shfl_down_sync(0xffffffffu, pm, o)); am = fmax(am, __shfl_down_sync(0xffffffffu, am, o)); }
    if ((threadIdx.x & 31) == 0) {
        atomicMax(out, (unsigned long long)__double_as_longlong(pm));
        atomicMax(out + 1, (unsigned long long)__double_as_longlong(am));
    }
}

// S = (P + P^T) / 2 into densities 0 .. nD-1 of out, A = (P - P^T) / 2 into nD .. 2 nD-1: the arithmetic of stage_host_density
__global__ void k_density_split(const double* __restrict__ P, double* __restrict__ out, int nD, int n) {
    const int64_t nn = (int64_t)n * n, total = nD * nn;
    for (int64_t x = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; x < total; x += (int64_t)gridDim.x * blockDim.x) {
        const int64_t d = x / nn, ij = x % nn;
        const int i = (int)(ij / n), j = (int)(ij % n);
        const double v = P[x], t = P[d * nn + (int64_t)j * n + i];
        out[x] = 0.5 * (v + t);
        out[total + x] = 0.5 * (v - t);
    }
}

// K[P] = K[S] + K[A] of a split stack: out = a + b, one FP64 add per element as in unstage_host_results
__global__ void k_add_into(double* __restrict__ out, const double* __restrict__ a, const double* __restrict__ b, size_t count) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) out[i] = a[i] + b[i];
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
static PairTableDev table_dev(const tuna_ctx* ctx) {
    PairTableDev T;
    T.pi = ctx->d_pi; T.pj = ctx->d_pj; T.cls = ctx->d_cls; T.npp = ctx->d_npp; T.ppoff = ctx->d_ppoff; T.pp = ctx->d_pp;
    for (int g = 0; g < 5; ++g) { T.gbeg[g] = ctx->pt.group_begin[g]; T.tbeg[g] = ctx->task_begin[g]; }
    return T;
}

static int grid_for(const tuna_ctx* ctx, int64_t work_items, int block, int per_sm) {
    int64_t want = (work_items + block - 1) / block;
    int64_t cap = (int64_t)ctx->sm_count * per_sm;
    if (want < 1) want = 1;
    return (int)std::min(want, cap);
}

// F(a,b) of SURVEY.md section 8(d): flops of the reference algorithm per primitive quartet.
static double reference_flops(int cls_a, int cls_b) {
    const int lxa = cls_a & 255, lya = (cls_a >> 8) & 255, lza = cls_a >> 16;
    const int lxb = cls_b & 255, lyb = (cls_b >> 8) & 255, lzb = cls_b >> 16;
    const int Nmax = lxa + lya + lza + lxb + lyb + lzb, Vmax = lza + lzb;
    const double nx = (lxa / 2 + 1) * (lxb / 2 + 1), nxy = nx * (lya / 2 + 1) * (lyb / 2 + 1), nzz = (lza + 1) * (lzb + 1);
    double rt = Nmax + 1;
    for (int v = 1; v <= Vmax; ++v) rt += (Nmax - v + 1) * (v == 1 ? 1 : 3);
    return 6 + 32 + 3 * Nmax + (Nmax + 1) + rt + 2 * nx + 3 * nxy + 5 * nxy * nzz + 8;
}

static void count_work(tuna_ctx* ctx) {
    const PairTable& T = ctx->pt;
    const int64_t np = T.npair;
    ctx->n_unique = np * (np + 1) / 2;
    ctx->n_surviving = 0; ctx->n_primq = 0; ctx->alg_eri_flops = 0;
    ctx->task_begin[0] = 0;
    for (int g = 0; g < 4; ++g) {
        const int64_t ng = T.group_begin[g + 1] - T.group_begin[g];
        ctx->task_begin[g + 1] = ctx->task_begin[g] + ng * (ng + 1) / 2;
        std::map<std::pair<int, int>, int64_t> hist;   // (class, npp) -> count
        for (int64_t a = T.group_begin[g]; a < T.group_begin[g + 1]; ++a) hist[{T.cls[a], T.npp[a]}]++;
        std::vector<std::pair<std::pair<int, int>, int64_t>> keys(hist.begin(), hist.end());
        for (size_t x = 0; x < keys.size(); ++x)
            for (size_t y = 0; y <= x; ++y) {
                const double cnt = (x == y) ? (double)keys[x].second * (keys[x].second + 1) / 2 : (double)keys[x].second * keys[y].second;
                const double primq = cnt * keys[x].first.second * keys[y].first.second;
                ctx->n_primq += (int64_t)primq;
                ctx->alg_eri_flops += primq * reference_flops(keys[x].first.first, keys[y].first.first);
            }
    }
    ctx->n_surviving = ctx->task_begin[4];
    ctx->alg_digest_flops = 12.0 * (double)ctx->n_surviving;
}

static int build_csr(tuna_ctx* ctx, CsrDev& M, int rows, int cols, const std::vector<double>& dense) {
    std::vector<int> rowptr(rows + 1, 0), col;
    std::vector<double> val;
    for (int r = 0; r < rows; ++r) {
        for (int c = 0; c < cols; ++c) {
            const double v = dense[(size_t)r * cols + c];
            if (v != 0.0) { col.push_back(c); val.push_back(v); }
        }
        rowptr[r + 1] = (int)col.size();
    }
    M.rows = rows; M.cols = cols;
    GROW(M.rowptr, rowptr.size());
    GROW(M.col, std::max<size_t>(col.size(), 1));
    GROW(M.val, std::max<size_t>(val.size(), 1));
    CK(cudaMemcpyAsync(M.rowptr, rowptr.data(), rowptr.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    if (!col.empty()) {
        CK(cudaMemcpyAsync(M.col, col.data(), col.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(M.val, val.data(), val.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return TUNA_OK;
}

static int rotate(tuna_ctx* ctx, const CsrDev& M, const double* in, double* out, int64_t outer, int64_t inner) {
    const int64_t total = outer * M.rows * inner;
    if (total == 0) return TUNA_OK;
    if (inner >= 128) {
        const int64_t rows = outer * M.rows;
        if (rows > 0x7fffffffLL) FAIL(TUNA_ERR_ARG, "rotate: tensor too large");
        const int ytiles = (int)std::min<int64_t>((inner + 1023) / 1024, 65535);       // up to four elements per thread
        k_rotate_axis_wide<<<dim3((unsigned)rows, (unsigned)ytiles), 256, 0, ctx->stream>>>(in, out, M.rowptr, M.col, M.val, M.cols, M.rows, inner);
    } else {
        const int threads = (int)std::min<int64_t>(256, ((int64_t)M.rows * inner + 31) / 32 * 32);
        const int64_t blocks = std::min<int64_t>(outer, (int64_t)ctx->sm_count * 64);
        k_rotate_axis_narrow<<<(unsigned)blocks, threads, 0, ctx->stream>>>(in, out, M.rowptr, M.col, M.val, outer, M.cols, M.rows, (int)inner);
    }
    ctx->launches++;
    CK(cudaGetLastError());
    return TUNA_OK;
}

static int ensure_mats(tuna_ctx* ctx, int nD, int n, int ncart) {
    const size_t need = (size_t)nD * n * n;
    GROW(ctx->d_P, need);
    GROW(ctx->d_J, need);
    GROW(ctx->d_K, need);
    const size_t needc = (size_t)nD * ncart * ncart;
    GROW(ctx->d_Pc, needc);
    GROW(ctx->d_Jc, needc);
    GROW(ctx->d_Kc, needc);
    GROW(ctx->d_tmp, needc);
    GROW(ctx->h_pin, 3 * need);
    return TUNA_OK;
}

// The AO-pair table (host build with OpenMP + one upload) on first use: ERI fill, Schwarz factors, direct J/K, work counters.
static int ensure_pairs(tuna_ctx* ctx) {
    if (ctx->pairs_ready) return TUNA_OK;
    if (ctx->ncart == 0) FAIL(TUNA_ERR_STATE, "call tuna_set_basis first");
    try {
        build_pair_table(ctx->hb, ctx->pt);
    } catch (const std::bad_alloc&) {
        FAIL(TUNA_ERR_NOMEM, "host allocation failed while building the pair table");
    }
    const PairTable& T = ctx->pt;
    GROW(ctx->d_pi, (size_t)T.npair);
    GROW(ctx->d_pj, (size_t)T.npair);
    GROW(ctx->d_cls, (size_t)T.npair);
    GROW(ctx->d_npp, (size_t)T.npair);
    GROW(ctx->d_ppoff, (size_t)T.npair);
    GROW(ctx->d_pp, T.pp.size());
    CK(cudaMemcpyAsync(ctx->d_pi, T.pi.data(), T.npair * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_pj, T.pj.data(), T.npair * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_cls, T.cls.data(), T.npair * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_npp, T.npp.data(), T.npair * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_ppoff, T.ppoff.data(), T.npair * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(ctx->d_pp, T.pp.data(), T.pp.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    count_work(ctx);
    ctx->pairs_ready = true;
    return TUNA_OK;
}

static int ensure_schwarz(tuna_ctx* ctx) {
    int rc;
    if ((rc = ensure_pairs(ctx))) return rc;
    if (ctx->d_Q) return TUNA_OK;
    DevBuf<double> Q;         // published only once its kernel is launched: d_Q != nullptr means "filled"
    GROW(Q, (size_t)ctx->pt.npair);
    k_schwarz<<<grid_for(ctx, ctx->pt.npair, 128, 16), 128, 0, ctx->stream>>>(table_dev(ctx), ctx->d_boys, ctx->d_herm, Q, ctx->pt.npair);
    ctx->launches++;
    CK(cudaGetLastError());
    ctx->d_Q = std::move(Q);
    return TUNA_OK;
}

extern "C" {

int tuna_ctx_create(int device, tuna_ctx** out) {
    if (!out) return TUNA_ERR_ARG;
    *out = nullptr;
    tuna_ctx* ctx = new (std::nothrow) tuna_ctx;
    if (!ctx) return TUNA_ERR_NOMEM;
    ctx->device = device;
    *out = ctx;   // returned even on failure so that tuna_last_error can be read; caller destroys it
    int ndev = 0;
    CK(cudaGetDeviceCount(&ndev));
    if (device < 0 || device >= ndev) FAIL(TUNA_ERR_ARG, "no such CUDA device: " + std::to_string(device));
    CK(cudaSetDevice(device));
    cudaDeviceProp prop;
    CK(cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    CK(cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking));
    ctx->stream = ctx->own_stream;
    for (int w = 0; w < 7; ++w)
        for (int s = 0; s < 2; ++s) CK(cudaEventCreate(&ctx->ev[w][s]));
    CK(cudaEventCreateWithFlags(&ctx->ev_group, cudaEventDisableTiming));
    for (int a = 0; a < tuna_ctx::NAUX; ++a) {
        CK(cudaStreamCreateWithFlags(&ctx->aux[a], cudaStreamNonBlocking));
        CK(cudaEventCreateWithFlags(&ctx->ev_join[a], cudaEventDisableTiming));
    }
    CK(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
    if (const char* ns = getenv("TUNA_B200_STREAMS")) ctx->naux = std::max(1, std::min((int)tuna_ctx::NAUX, atoi(ns)));
    std::vector<double> boys, herm;
    build_boys_table(boys);
    build_hermite_poly_table(herm);
    GROW(ctx->d_boys, boys.size());
    GROW(ctx->d_herm, herm.size());
    GROW(ctx->d_scalars, (size_t)4);
    CK(cudaMemcpy(ctx->d_boys, boys.data(), boys.size() * sizeof(double), cudaMemcpyHostToDevice));
    CK(cudaMemcpy(ctx->d_herm, herm.data(), herm.size() * sizeof(double), cudaMemcpyHostToDevice));
    CK(cudaMemset(ctx->d_scalars, 0, 4 * sizeof(unsigned long long)));
    return TUNA_OK;
}

int tuna_ctx_destroy(tuna_ctx* ctx) {
    if (!ctx) return TUNA_OK;
    cudaSetDevice(ctx->device);
    if (ctx->stream) cudaStreamSynchronize(ctx->stream);
    for (int w = 0; w < 7; ++w)
        for (int s = 0; s < 2; ++s) if (ctx->ev[w][s]) cudaEventDestroy(ctx->ev[w][s]);
    if (ctx->ev_group) cudaEventDestroy(ctx->ev_group);
    for (int a = 0; a < tuna_ctx::NAUX; ++a) {
        if (ctx->aux[a]) { cudaStreamSynchronize(ctx->aux[a]); cudaStreamDestroy(ctx->aux[a]); }
        if (ctx->ev_join[a]) cudaEventDestroy(ctx->ev_join[a]);
    }
    if (ctx->ev_fork) cudaEventDestroy(ctx->ev_fork);
    if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
    delete ctx;
    return TUNA_OK;
}

const char* tuna_last_error(const tuna_ctx* ctx) { return ctx ? ctx->err.c_str() : "null context"; }

int tuna_set_stream(tuna_ctx* ctx, void* s) {
    if (!ctx) return TUNA_ERR_ARG;
    ctx->stream = s ? (cudaStream_t)s : ctx->own_stream;
    return TUNA_OK;
}

int tuna_set_basis(tuna_ctx* ctx, int ncart, const double* origins_z, const int32_t* lmn, const int32_t* nprim, const int64_t* prim_offset,
                   const double* exps, const double* coef_eff) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (ncart <= 0 || !origins_z || !lmn || !nprim || !prim_offset || !exps || !coef_eff) FAIL(TUNA_ERR_ARG, "tuna_set_basis: null or empty basis");
    CK(cudaSetDevice(ctx->device));
    HostBasis& B = ctx->hb;
    B = HostBasis();
    B.ncart = ncart;
    int64_t total = 0;
    for (int i = 0; i < ncart; ++i) {
        if (nprim[i] <= 0) FAIL(TUNA_ERR_ARG, "tuna_set_basis: basis function without primitives");
        for (int c = 0; c < 3; ++c)
            if (lmn[3 * i + c] < 0 || lmn[3 * i + c] > 5) FAIL(TUNA_ERR_ARG, "tuna_set_basis: angular momentum outside 0..5 (only up to H functions, tuna_molecule.py:612-618)");
        if (lmn[3 * i] + lmn[3 * i + 1] + lmn[3 * i + 2] > 5) FAIL(TUNA_ERR_ARG, "tuna_set_basis: shell angular momentum above 5");
        total = std::max<int64_t>(total, prim_offset[i] + nprim[i]);
    }
    try {
        B.oz.assign(origins_z, origins_z + ncart);
        B.lmn.assign(lmn, lmn + 3 * (size_t)ncart);
        B.nprim.assign(nprim, nprim + ncart);
        B.off.assign(prim_offset, prim_offset + ncart);
        B.exps.assign(exps, exps + total);
        B.ceff.assign(coef_eff, coef_eff + total);
        for (int64_t k = 0; k < total; ++k)
            if (!(B.exps[k] > 0.0)) FAIL(TUNA_ERR_ARG, "tuna_set_basis: non-positive exponent");
    } catch (const std::bad_alloc&) {
        FAIL(TUNA_ERR_NOMEM, "host allocation failed while copying the basis");
    }
    ctx->ncart = ncart;
    ctx->basis_sum = checksum(B.oz.data(), B.oz.size() * sizeof(B.oz[0]), checksum(B.lmn.data(), B.lmn.size() * sizeof(B.lmn[0]),
                     checksum(B.nprim.data(), B.nprim.size() * sizeof(B.nprim[0]), checksum(B.off.data(), B.off.size() * sizeof(B.off[0]),
                     checksum(B.exps.data(), B.exps.size() * sizeof(B.exps[0]), checksum(B.ceff.data(), B.ceff.size() * sizeof(B.ceff[0])))))));
    ctx->U_sum = 0;
    ctx->pairs_ready = false;
    ctx->pt = PairTable();
    ctx->n_unique = ctx->n_surviving = ctx->n_primq = 0;
    ctx->d_Q.reset();
    ctx->d_eri_cart.reset();
    ctx->d_eri_sph.reset();
    ctx->n_stored = 0;
    ctx->nbf = 0;
    ctx->U_shell_blocks = false;
    build_shell_tab(ctx->stab);
    ctx->shell_ready = false;
    drop_store(ctx);
    ctx->jobsets4.clear();
    ctx->cur_jobset4 = -1;
    detect_shells(ctx->hb, ctx->stab, ctx->ss);     // ss.ok == false -> direct mode uses the per-component kernel
    const char* eng = getenv("TUNA_B200_DIRECT_ENGINE");
    ctx->direct_engine = (eng && std::string(eng) == "generic") ? 0 : 1;
    return TUNA_OK;
} TUNA_CATCH

int tuna_set_transform(tuna_ctx* ctx, int nbf, const double* U) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (ctx->ncart == 0) FAIL(TUNA_ERR_STATE, "tuna_set_transform: call tuna_set_basis first");
    if (nbf <= 0 || !U) FAIL(TUNA_ERR_ARG, "tuna_set_transform: bad arguments");
    CK(cudaSetDevice(ctx->device));
    drop_store(ctx);
    const int nc = ctx->ncart;
    std::vector<double> u(U, U + (size_t)nbf * nc), ut((size_t)nc * nbf);
    for (int p = 0; p < nbf; ++p)
        for (int a = 0; a < nc; ++a) ut[(size_t)a * nbf + p] = u[(size_t)p * nc + a];
    int rc;
    if ((rc = build_csr(ctx, ctx->U, nbf, nc, u))) return rc;
    if ((rc = build_csr(ctx, ctx->Ut, nc, nbf, ut))) return rc;
    if (ctx->ss.ok) {
        std::vector<double> uf(u), uft(ut);
        for (int p = 0; p < nbf; ++p)
            for (int a = 0; a < nc; ++a) {
                uf[(size_t)p * nc + a] *= ctx->ss.fnorm[a];
                uft[(size_t)a * nbf + p] *= ctx->ss.fnorm[a];
            }
        if ((rc = build_csr(ctx, ctx->Uf, nbf, nc, uf))) return rc;
        if ((rc = build_csr(ctx, ctx->Uft, nc, nbf, uft))) return rc;
    }
    ctx->nbf = nbf;
    ctx->U_sum = checksum(u.data(), u.size() * sizeof(double), (uint64_t)nbf);
    ctx->U_identity = (nbf == nc);
    for (int p = 0; p < nbf && ctx->U_identity; ++p)
        for (int a = 0; a < nc; ++a)
            if (u[(size_t)p * nc + a] != (p == a ? 1.0 : 0.0)) { ctx->U_identity = false; break; }
    ctx->U_shell_blocks = false;
    SphShells Y;
    if (build_sph_shells(ctx->ss, ctx->stab, nbf, nc, u.data(), Y)) {
        GROW(ctx->d_sph_n, Y.nsph.size());
        GROW(ctx->d_sph_idx, Y.sph.size());
        GROW(ctx->d_sph_uoff, Y.uoff.size());
        GROW(ctx->d_sph_par, Y.par.size());
        GROW(ctx->d_sph_u, std::max<size_t>(Y.u.size(), 1));
        CK(cudaMemcpyAsync(ctx->d_sph_n, Y.nsph.data(), Y.nsph.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_sph_idx, Y.sph.data(), Y.sph.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_sph_uoff, Y.uoff.data(), Y.uoff.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_sph_par, Y.par.data(), Y.par.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_sph_u, Y.u.data(), Y.u.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->U_shell_blocks = true;
    }
    return TUNA_OK;
} TUNA_CATCH

// The dense tensor is filled by the shell-quartet engine (rather than k_eri_fill) for a basis that groups into shells and has contracted
// shells, unless TUNA_B200_DIRECT_ENGINE=generic; TUNA_B200_FILL_ENGINE=1 / 0 forces the choice (reasons in tuna_eri_fill_cart).
static bool fill_uses_engine(const tuna_ctx* ctx) {
    bool contracted = false;
    for (const auto& sh : ctx->ss.shells) contracted = contracted || sh.nprim > 1;
    const char* ef = getenv("TUNA_B200_FILL_ENGINE");
    return ctx->direct_engine == 1 && ctx->ss.ok && (ef ? atoi(ef) != 0 : contracted);
}

int tuna_eri_fill_cart(tuna_ctx* ctx) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (ctx->ncart == 0) FAIL(TUNA_ERR_STATE, "tuna_eri_fill_cart: call tuna_set_basis first");
    CK(cudaSetDevice(ctx->device));
    const size_t n = ctx->ncart, count = n * n * n * n;
    int rc;
    if ((rc = ensure_pairs(ctx))) return rc;
    // A basis that groups into shells AND has contracted shells is filled by the shell-quartet engine (shell4.cuh, fill mode: Boys values, R,
    // the x/y table and the z contractions are shared by all components of a shell quartet, contracted quartets are split over work items)
    // followed by the scatter pass; an uncontracted basis keeps the per-AO-quartet kernel, which is as fast there (ET100: 1.40 vs 1.52 ms;
    // N2/cc-pVTZ: 3.7 vs 0.87 ms, Ne2/cc-pVQZ: 13.6 vs 5.4 ms).  TUNA_B200_FILL_ENGINE=1 / 0 forces one or the other.  Both leave the same
    // tensor: one value written to all eight images, exact zeros for the parity-forbidden elements.
    bool engine = fill_uses_engine(ctx);
    // the dense tensor is never sharded (every rank holds all of it): the fill runs as rank 0 of 1, whatever tuna_set_shard said
    struct ShardGuard { tuna_ctx* c; int r, n; ~ShardGuard() { c->shard_rank = r; c->shard_n = n; } } guard{ctx, ctx->shard_rank, ctx->shard_n};
    GROW(ctx->d_eri_cart, count);
    if (engine) {
        ctx->shard_rank = 0; ctx->shard_n = 1;
        rc = ensure_shell4(ctx, 0.0, 0);
        if (rc) {       // when only the scratch rows did not fit, the per-AO-quartet kernel (no scratch) takes over
            if (rc != TUNA_ERR_NOMEM) return rc;
            engine = false;
        }
    }
    CK(cudaMemsetAsync(ctx->d_eri_cart, 0, count * sizeof(double), ctx->stream));
    CK(cudaEventRecord(ctx->ev[0][0], ctx->stream));
    if (engine) {
        const tuna_ctx::JobSet4& JS = ctx->jobsets4[ctx->cur_jobset4];
        if ((rc = launch_shell4_jobs(ctx, 0, nullptr, nullptr, nullptr, nullptr, 0.0, 0))) return rc;
        if (JS.scatter_total > 0) {
            ShellData D;
            D.pairA = ctx->d_pairA; D.pairB = ctx->d_pairB; D.pair_rec = ctx->d_pair_rec; D.rec = ctx->d_rec; D.pairQ = ctx->d_pairQ;
            D.sh_ao = ctx->d_sh_ao; D.boys = ctx->d_boys; D.herm = ctx->d_herm; D.fix_lo = 0;
            k_fill_scatter<<<(unsigned)std::min<long long>(JS.scatter_total, (long long)ctx->sm_count * 64), 256, 0, ctx->stream>>>(JS.d_all_jobs, JS.d_scatter_pre, (int)JS.jobs.size(), D, ctx->d_fnorm,
                                                                                            ctx->d_eri_cart, ctx->ncart);
            ctx->launches++;
        }
    } else {
        k_eri_fill<<<grid_for(ctx, ctx->task_begin[4], 128, 16), 128, 0, ctx->stream>>>(table_dev(ctx), ctx->d_boys, ctx->d_herm, ctx->d_eri_cart, ctx->ncart);
        ctx->launches++;
    }
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev[0][1], ctx->stream));
    if (engine) {       // the scratch rows (the unique integrals once per primitive chunk) are only needed until the scatter pass has run
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->jobsets4.erase(ctx->jobsets4.begin() + ctx->cur_jobset4);
        ctx->cur_jobset4 = -1;
    }
    return TUNA_OK;
} TUNA_CATCH

int tuna_eri_cart_to_sph(tuna_ctx* ctx, int keep_cart) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (!ctx->d_eri_cart) FAIL(TUNA_ERR_STATE, "tuna_eri_cart_to_sph: no Cartesian tensor resident (call tuna_eri_fill_cart)");
    if (ctx->nbf == 0) FAIL(TUNA_ERR_STATE, "tuna_eri_cart_to_sph: call tuna_set_transform first");
    CK(cudaSetDevice(ctx->device));
    const int64_t nc = ctx->ncart, nb = ctx->nbf;
    int rc;
    ctx->d_eri_sph.reset();
    ctx->n_stored = 0;
    CK(cudaEventRecord(ctx->ev[1][0], ctx->stream));
    if (ctx->U_identity) {   // CARTHARM: no rotation (tuna_kernel.py:481-483)
        if (keep_cart) {
            GROW(ctx->d_eri_sph, (size_t)(nc * nc * nc * nc));
            CK(cudaMemcpyAsync(ctx->d_eri_sph, ctx->d_eri_cart, (size_t)(nc * nc * nc * nc) * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
        } else {
            ctx->d_eri_sph = std::move(ctx->d_eri_cart);
        }
        CK(cudaEventRecord(ctx->ev[1][1], ctx->stream));
        ctx->n_stored = (int)nc;
        ctx->eri_pair_sym = true;          // the fill scatters one value to all eight images
        return TUNA_OK;
    }
    // Four single-index passes ping-ponging between two work buffers; every allocation happens before the timed region and nothing
    // synchronises inside it (stream order is enough).  Without keep_cart the Cartesian tensor's own storage is the second buffer.
    DevBuf<double> t1, t2;
    GROW(t1, (size_t)(nb * nc * nc * nc));
    if (keep_cart) GROW(t2, (size_t)(nb * nb * nc * nc));
    GROW(ctx->d_eri_sph, (size_t)(nb * nb * nb * nb));
    double* w2 = keep_cart ? t2.get() : ctx->d_eri_cart.get();
    CK(cudaEventRecord(ctx->ev[1][0], ctx->stream));
    rc = rotate(ctx, ctx->U, ctx->d_eri_cart, t1, 1, nc * nc * nc);
    if (!rc) rc = rotate(ctx, ctx->U, t1, w2, nb, nc * nc);
    if (!rc) rc = rotate(ctx, ctx->U, w2, t1, nb * nb, nc);
    if (!rc) rc = rotate(ctx, ctx->U, t1, ctx->d_eri_sph, nb * nb * nb, 1);
    if (!rc) { CK(cudaEventRecord(ctx->ev[1][1], ctx->stream)); }
    cudaStreamSynchronize(ctx->stream);
    if (!keep_cart) ctx->d_eri_cart.reset();
    if (rc) { ctx->d_eri_sph.reset(); return rc; }
    ctx->n_stored = (int)nb;
    return check_pair_symmetry(ctx);
} TUNA_CATCH

int tuna_eri_fill_sph(tuna_ctx* ctx) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (ctx->ncart == 0) FAIL(TUNA_ERR_STATE, "tuna_eri_fill_sph: call tuna_set_basis first");
    if (ctx->nbf == 0) FAIL(TUNA_ERR_STATE, "tuna_eri_fill_sph: call tuna_set_transform first");
    CK(cudaSetDevice(ctx->device));
    int rc;
    if ((rc = ensure_pairs(ctx))) return rc;
    // Bases the engine does not fill, a U that is not block-diagonal over the engine's shells, and CARTHARM (identity U, the Cartesian
    // tensor is adopted) take the two-step path; so does a fill whose scratch rows do not fit (tuna_eri_fill_cart then uses k_eri_fill).
    const auto two_step = [ctx]() { const int r = tuna_eri_fill_cart(ctx); return r ? r : tuna_eri_cart_to_sph(ctx, 0); };
    if (!fill_uses_engine(ctx) || !ctx->U_shell_blocks || ctx->U_identity) return two_step();
    ctx->d_eri_cart.reset();
    ctx->d_eri_sph.reset();
    ctx->n_stored = 0;
    const size_t nb = ctx->nbf;
    struct ShardGuard { tuna_ctx* c; int r, n; ~ShardGuard() { c->shard_rank = r; c->shard_n = n; } } guard{ctx, ctx->shard_rank, ctx->shard_n};
    ctx->shard_rank = 0; ctx->shard_n = 1;
    GROW(ctx->d_eri_sph, nb * nb * nb * nb);
    rc = ensure_shell4(ctx, 0.0, 0);
    if (rc) {
        ctx->d_eri_sph.reset();
        if (rc != TUNA_ERR_NOMEM) return rc;
        return two_step();
    }
    const size_t js = (size_t)ctx->cur_jobset4;
    // the fill job set holds the scratch rows: it is dropped after the pass, and on every error path with the half-built tensor
    const auto fail = [ctx](int code) {
        cudaStreamSynchronize(ctx->stream);
        ctx->jobsets4.erase(ctx->jobsets4.begin() + ctx->cur_jobset4);
        ctx->cur_jobset4 = -1;
        ctx->d_eri_sph.reset();
        return code;
    };
    // per-CTA Cartesian block (global, L2 resident) and contraction buffers (shared): sized by the largest class of the job set
    long long blk = 1, xsz = 1;
    for (const auto& jh : ctx->jobsets4[js].jobs) {
        const long long nB = sph_ncart(jh.job.Lb), ncd = (long long)sph_ncart(jh.job.Lc) * sph_ncart(jh.job.Ld);
        blk = std::max(blk, sph_ncart(jh.job.La) * nB * ncd);
        xsz = std::max(xsz, nB * ncd);
    }
    xsz = (xsz + 1) & ~1LL;
    const long long total = ctx->jobsets4[js].scatter_total;
    const long long ws_cap = 64ll << 20;       // bytes of Cartesian blocks: at least one CTA per SM, at most four
    const long long grid = std::max<long long>(1, std::min<long long>(total, std::max<long long>(ctx->sm_count, std::min<long long>(4ll * ctx->sm_count, ws_cap / (8 * blk)))));
    DevBuf<double> ws;
    if (const int g = ws.grow((size_t)(grid * blk), ctx->err)) return fail(g);
    const size_t smem = (size_t)(2 * xsz) * sizeof(double);
    if (smem > 48 * 1024) {
        if (const cudaError_t e = opt_in_smem<k_fill_scatter_sph>(ctx)) { ctx->err = cudaGetErrorString(e); return fail(TUNA_ERR_CUDA); }
    }
    CK(cudaEventRecord(ctx->ev[0][0], ctx->stream));
    if ((rc = launch_shell4_jobs(ctx, 0, nullptr, nullptr, nullptr, nullptr, 0.0, 0))) return fail(rc);
    if (total > 0) {
        const tuna_ctx::JobSet4& JS = ctx->jobsets4[js];
        ShellData D;
        D.pairA = ctx->d_pairA; D.pairB = ctx->d_pairB; D.pair_rec = ctx->d_pair_rec; D.rec = ctx->d_rec; D.pairQ = ctx->d_pairQ;
        D.sh_ao = ctx->d_sh_ao; D.boys = ctx->d_boys; D.herm = ctx->d_herm; D.fix_lo = 0;
        SphData Y;
        Y.nsph = ctx->d_sph_n; Y.sph = ctx->d_sph_idx; Y.uoff = ctx->d_sph_uoff; Y.u = ctx->d_sph_u; Y.par = ctx->d_sph_par;
        k_fill_scatter_sph<<<(unsigned)grid, 256, smem, ctx->stream>>>(JS.d_all_jobs, JS.d_scatter_pre, (int)JS.jobs.size(), D, Y, ctx->d_fnorm, ws, blk,
                                                                       (int)xsz, ctx->d_eri_sph, (int)nb);
        ctx->launches++;
    }
    cudaError_t le = cudaGetLastError();
    if (le == cudaSuccess) le = cudaEventRecord(ctx->ev[0][1], ctx->stream);
    if (le == cudaSuccess) le = cudaStreamSynchronize(ctx->stream);
    if (le != cudaSuccess) { ctx->err = cudaGetErrorString(le); return fail(TUNA_ERR_CUDA); }
    ctx->jobsets4.erase(ctx->jobsets4.begin() + ctx->cur_jobset4);      // the scratch rows are only needed until the pass has run
    ctx->cur_jobset4 = -1;
    ctx->n_stored = (int)nb;
    ctx->eri_pair_sym = true;          // one value is written to all eight images
    return TUNA_OK;
} TUNA_CATCH

int tuna_eri_download(tuna_ctx* ctx, int which, double* host_out) try {
    if (!ctx || !host_out) return TUNA_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const double* src = which == 0 ? ctx->d_eri_cart : ctx->d_eri_sph;
    const size_t n = which == 0 ? ctx->ncart : ctx->n_stored;
    if (!src) FAIL(TUNA_ERR_STATE, "tuna_eri_download: requested tensor is not resident");
    CK(cudaMemcpyAsync(host_out, src, n * n * n * n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TUNA_OK;
} TUNA_CATCH

int tuna_eri_upload(tuna_ctx* ctx, int n, const double* host_in) try {
    if (!ctx || !host_in || n <= 0) return TUNA_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    const size_t count = (size_t)n * n * n * n;
    ctx->n_stored = 0;
    ctx->d_eri_sph.reset();
    GROW(ctx->d_eri_sph, count);
    CK(cudaMemcpyAsync(ctx->d_eri_sph, host_in, count * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    ctx->n_stored = n;
    return check_pair_symmetry(ctx);
} TUNA_CATCH

int tuna_eri_single(tuna_ctx* ctx, int i, int j, int k, int l, double* out) try {
    if (!ctx || !out) return TUNA_ERR_ARG;
    const int n = ctx->ncart;
    if (n == 0) FAIL(TUNA_ERR_STATE, "tuna_eri_single: call tuna_set_basis first");
    if (i < 0 || j < 0 || k < 0 || l < 0 || i >= n || j >= n || k >= n || l >= n) FAIL(TUNA_ERR_ARG, "tuna_eri_single: index out of range");
    CK(cudaSetDevice(ctx->device));
    const HostBasis& B = ctx->hb;
    auto cls_of = [&](int a, int b) {
        return (B.lmn[3 * a] + B.lmn[3 * b]) | ((B.lmn[3 * a + 1] + B.lmn[3 * b + 1]) << 8) | ((B.lmn[3 * a + 2] + B.lmn[3 * b + 2]) << 16);
    };
    const int cA = cls_of(i, j), cB = cls_of(k, l);
    if ((((cA & 255) + (cB & 255)) & 1) || ((((cA >> 8) & 255) + ((cB >> 8) & 255)) & 1)) { *out = 0.0; return TUNA_OK; }   // pyx:1397-1400
    const int nA = B.nprim[i] * B.nprim[j], nB = B.nprim[k] * B.nprim[l];
    std::vector<double> rec((size_t)(nA + nB) * PP_DOUBLES), scratch;
    double* r = rec.data();
    for (int a = 0; a < B.nprim[i]; ++a)
        for (int b = 0; b < B.nprim[j]; ++b, r += PP_DOUBLES) fill_prim_record(r, B, i, j, B.off[i] + a, B.off[j] + b, scratch);
    for (int a = 0; a < B.nprim[k]; ++a)
        for (int b = 0; b < B.nprim[l]; ++b, r += PP_DOUBLES) fill_prim_record(r, B, k, l, B.off[k] + a, B.off[l] + b, scratch);
    DevBuf<double> d;
    GROW(d, rec.size() + 1);
    CK(cudaMemcpyAsync(d + 1, rec.data(), rec.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    k_eri_single<<<1, 32, 0, ctx->stream>>>(d + 1, nA, cA, d + 1 + (size_t)nA * PP_DOUBLES, nB, cB, ctx->d_boys, ctx->d_herm, d);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(out, d, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TUNA_OK;
} TUNA_CATCH

int tuna_schwarz(tuna_ctx* ctx, double* host_out) try {
    if (!ctx || !host_out) return TUNA_ERR_ARG;
    if (ctx->ncart == 0) FAIL(TUNA_ERR_STATE, "tuna_schwarz: call tuna_set_basis first");
    CK(cudaSetDevice(ctx->device));
    int rc;
    if ((rc = ensure_schwarz(ctx))) return rc;
    std::vector<double> q((size_t)ctx->pt.npair);
    CK(cudaMemcpyAsync(q.data(), ctx->d_Q, q.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    const int n = ctx->ncart;
    for (int64_t a = 0; a < ctx->pt.npair; ++a) {
        host_out[(size_t)ctx->pt.pi[a] * n + ctx->pt.pj[a]] = q[a];
        host_out[(size_t)ctx->pt.pj[a] * n + ctx->pt.pi[a]] = q[a];
    }
    return TUNA_OK;
} TUNA_CATCH

}  // extern "C"

// Does the stored tensor have the pair-exchange symmetry (il|kj) = (kj|il) to rounding?  (Any physical ERI tensor does; an
// arbitrary uploaded array need not, and then the general kernels are used.)
static int check_pair_symmetry(tuna_ctx* ctx) {
    ctx->eri_pair_sym = false;
    if (!ctx->d_eri_sph || ctx->n_stored == 0) return TUNA_OK;
    const int n = ctx->n_stored;
    CK(cudaMemsetAsync(ctx->d_scalars + 2, 0, 2 * sizeof(unsigned long long), ctx->stream));
    k_pair_sym_check<<<grid_for(ctx, (int64_t)n * n * n * n, 256, 8), 256, 0, ctx->stream>>>(ctx->d_eri_sph, n, ctx->d_scalars + 2);
    ctx->launches++;
    CK(cudaGetLastError());
    unsigned long long h[2];
    CK(cudaMemcpyAsync(h, ctx->d_scalars + 2, sizeof(h), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    double md, mx;
    std::memcpy(&md, &h[0], 8); std::memcpy(&mx, &h[1], 8);
    ctx->eri_pair_sym = md <= 1e-13 * mx;
    return TUNA_OK;
}

template <int ND, int MT>
static cudaError_t launch_jk_sym(tuna_ctx* ctx, const double* P, double* Jpart, double* Kslot, int* Krow, int n, int r, int nstage, int kslots,
                                 int ncons, int grid, size_t smem) {
    if (cudaError_t e = opt_in_smem<k_jk_stored_sym<ND, MT>>(ctx); e != cudaSuccess) return e;
    k_jk_stored_sym<ND, MT><<<grid, ncons + 32, smem, ctx->stream>>>(ctx->d_eri_sph, P, Jpart, Kslot, Krow, n, r, nstage, kslots, ncons);
    return cudaGetLastError();
}

// Symmetric streaming path; returns TUNA_OK with *done = false when the shape does not fit its register / shared-memory budget.
static int jk_stored_sym(tuna_ctx* ctx, int nD, const double* dP, double* dJ, double* dK, bool* done) {
    *done = false;
    const int n = ctx->n_stored;
    const size_t nn = (size_t)n * n;
    if (!ctx->eri_pair_sym || (n & 1) || n < 16 || n > 960) return TUNA_OK;
    const int r = std::min(n, 960 / n), T = r * n, ncons = (T + 31) / 32 * 32;
    const int mt_need = (n + r - 1) / r;
    const int MT = mt_need <= 4 ? 4 : mt_need <= 8 ? 8 : mt_need <= 16 ? 16 : 0;
    const int nd_max = MT == 4 ? 4 : MT == 8 ? 2 : MT == 16 ? 1 : 0;
    if (MT == 0 || (nD + nd_max - 1) / nd_max > (nD + 3) / 4) return TUNA_OK;      // never more passes over the tensor than the general kernel
    const int grid = (int)std::min<long long>((long long)ctx->sm_count, (long long)nn);
    const int kslots = (int)((nn / grid + 1 + n - 1) / n) + 2;
    const int nslots = grid * kslots;
    for (int d0 = 0; d0 < nD; d0 += nd_max) {
        const int nd = std::min(nd_max, nD - d0);
        const size_t fixed = ((size_t)nd * nn + (size_t)2 * nd * r * n) * sizeof(double) + 2 * 16 * sizeof(uint64_t) + 128;
        const size_t tile_bytes = (size_t)2 * T * sizeof(double);
        if (fixed + 4 * tile_bytes > 227 * 1024) return d0 == 0 ? TUNA_OK : TUNA_ERR_STATE;
        const int nstage = (int)std::min<size_t>(16, (227 * 1024 - fixed) / tile_bytes);
        const size_t smem = (size_t)nstage * tile_bytes + fixed;
        // workspace: Kslot rows | Krow tags | Jpart
        const size_t o_krow = (size_t)nslots * nd_max * n, o_jpart = o_krow + (size_t)(nslots + 1) / 2 + 2;
        GROW(ctx->d_Kpart, o_jpart + (size_t)grid * nd_max * nn);
        double* Kslot = ctx->d_Kpart;
        int* Krow = reinterpret_cast<int*>(ctx->d_Kpart + o_krow);
        double* Jpart = ctx->d_Kpart + o_jpart;
        const double* P = dP + d0 * nn;
        if (d0 == 0) CK(cudaEventRecord(ctx->ev[2][0], ctx->stream));
        cudaError_t e = cudaErrorInvalidValue;
#define TUNA_SYM(NDV, MTV) e = launch_jk_sym<NDV, MTV>(ctx, P, Jpart, Kslot, Krow, n, r, nstage, kslots, ncons, grid, smem)
        if (MT == 4) { switch (nd) { case 1: TUNA_SYM(1, 4); break; case 2: TUNA_SYM(2, 4); break; case 3: TUNA_SYM(3, 4); break; default: TUNA_SYM(4, 4); break; } }
        else if (MT == 8) { if (nd == 1) TUNA_SYM(1, 8); else TUNA_SYM(2, 8); }
        else TUNA_SYM(1, 16);
#undef TUNA_SYM
        ctx->launches++;
        if (e != cudaSuccess) FAIL(TUNA_ERR_CUDA, std::string("k_jk_stored_sym launch: ") + cudaGetErrorString(e));
        {
            static const bool pdl = getenv("TUNA_B200_PDL") && atoi(getenv("TUNA_B200_PDL")) == 1;     // opt-in: measured slightly slower (36.9 vs 40.1 us at nbf 60)
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3((unsigned)(((int64_t)nd * nn * 8 + 255) / 256));
            cfg.blockDim = dim3(256);
            cfg.stream = ctx->stream;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
            at[0].val.programmaticStreamSerializationAllowed = 1;
            cfg.attrs = at;
            cfg.numAttrs = pdl ? 1 : 0;
            const double* jp = Jpart; const double* ks = Kslot; const int* kr = Krow;
            double* jo = dJ ? dJ + d0 * nn : nullptr; double* ko = dK ? dK + d0 * nn : nullptr;
            CK(cudaLaunchKernelEx(&cfg, k_sym_reduce, jp, jo, ks, kr, ko, nd, n, grid, kslots));
        }
        ctx->launches++;
    }
    CK(cudaEventRecord(ctx->ev[2][1], ctx->stream));
    *done = true;
    return TUNA_OK;
}

template <int ND>
static cudaError_t launch_jk_tma(tuna_ctx* ctx, const double* P, double* J, double* Kslot, int* Krow, int n, int r, int R, int q, int nstage,
                                 int kslots, int grid, int threads, size_t smem) {
    if (cudaError_t e = opt_in_smem<k_jk_stored_tma<ND>>(ctx); e != cudaSuccess) return e;
    k_jk_stored_tma<ND><<<grid, threads, smem, ctx->stream>>>(ctx->d_eri_sph, P, J, Kslot, Krow, n, r, R, q, nstage, kslots);
    return cudaGetLastError();
}

extern "C" int tuna_jk_stored_dev(tuna_ctx* ctx, int nD, const double* dP, double* dJ, double* dK) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (!ctx->d_eri_sph || ctx->n_stored == 0) FAIL(TUNA_ERR_STATE, "tuna_jk_stored: no stored tensor resident");
    if (nD <= 0 || !dP) FAIL(TUNA_ERR_ARG, "tuna_jk_stored: bad arguments");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n_stored;
    if (n > 1024) FAIL(TUNA_ERR_ARG, "tuna_jk_stored: stored mode supports n <= 1024");
    int rc;
    const size_t nn = (size_t)n * n;
    const char* env_k = getenv("TUNA_B200_STORED_KERNEL");
    const bool want_tma = !(env_k && std::string(env_k) == "simple");
    if (!env_k || std::string(env_k) == "sym") {
        bool done = false;
        if ((rc = jk_stored_sym(ctx, nD, dP, dJ, dK, &done))) return rc;
        if (done) return TUNA_OK;
    }
    if (want_tma && (n % 2 == 0) && n >= 8) {
        // ---- TMA-streamed persistent kernel (16-byte alignment of every row tile needs an even n) ----
        const int r = std::max(1, 512 / n);
        const int threads = (n * r + 31) / 32 * 32;
        const int nwarp = threads / 32;
        const char* env_tile = getenv("TUNA_B200_JK_TILE_KB");
        const char* env_st = getenv("TUNA_B200_JK_STAGES");
        const char* env_cps = getenv("TUNA_B200_JK_CTAS_PER_SM");
        // knobs are clamped to what the kernel can run: a zero tile would divide by zero, zero stages would leave the consumers waiting
        // on an mbarrier no copy ever completes, zero CTAs per SM an empty grid, and a ring larger than 227 KB would not launch
        const size_t tile_budget = (size_t)(env_tile ? std::min(64, std::max(1, atoi(env_tile))) : 24) * 1024;
        int q = (int)((nn * sizeof(double) + tile_budget - 1) / tile_budget);
        int R = (n + q - 1) / q;
        R = (R + r - 1) / r * r;                       // whole row groups per tile
        q = (n + R - 1) / R;
        int nstage = env_st ? std::max(1, std::min(atoi(env_st), JK_MAX_STAGES)) : 3;
        const size_t smem_fixed = (2 * (size_t)nwarp * 4 + (size_t)4 * r * n) * sizeof(double) + JK_MAX_STAGES * sizeof(uint64_t) + 16;
        while (nstage > 1 && (size_t)nstage * R * n * sizeof(double) + smem_fixed > 227 * 1024) --nstage;
        const long long total = (long long)n * n;
        const int grid = (int)std::min<long long>((long long)ctx->sm_count * (env_cps ? std::max(1, atoi(env_cps)) : 2), total);
        const int kslots = (int)((total / grid + 1 + n - 1) / n) + 2;
        const int nslots = grid * kslots;
        const size_t need_kpart = (size_t)nslots * 4 * n + (size_t)(nslots + 1) / 2 + 8;       // doubles: partial rows + row tags
        if (dK) GROW(ctx->d_Kpart, need_kpart);
        CK(cudaEventRecord(ctx->ev[2][0], ctx->stream));
        for (int d0 = 0; d0 < nD; d0 += 4) {
            const int nd = std::min(4, nD - d0);
            if (!dK) GROW(ctx->d_Kpart, need_kpart);      // K not requested: the kernel still needs scratch rows
            double* Kslot = ctx->d_Kpart;
            int* Krow = reinterpret_cast<int*>(ctx->d_Kpart + (size_t)nslots * 4 * n);
            CK(cudaMemsetAsync(Krow, 0xFF, (size_t)nslots * sizeof(int), ctx->stream));
            const size_t smem = ((size_t)nstage * R * n + 2 * (size_t)nwarp * nd + (size_t)nd * r * n) * sizeof(double) + JK_MAX_STAGES * sizeof(uint64_t) + 16;
            const double* P = dP + d0 * nn;
            double* J = dJ ? dJ + d0 * nn : nullptr;
            cudaError_t e;
            switch (nd) {
                case 1: e = launch_jk_tma<1>(ctx, P, J, Kslot, Krow, n, r, R, q, nstage, kslots, grid, threads, smem); break;
                case 2: e = launch_jk_tma<2>(ctx, P, J, Kslot, Krow, n, r, R, q, nstage, kslots, grid, threads, smem); break;
                case 3: e = launch_jk_tma<3>(ctx, P, J, Kslot, Krow, n, r, R, q, nstage, kslots, grid, threads, smem); break;
                default: e = launch_jk_tma<4>(ctx, P, J, Kslot, Krow, n, r, R, q, nstage, kslots, grid, threads, smem); break;
            }
            ctx->launches++;
            if (e != cudaSuccess) FAIL(TUNA_ERR_CUDA, std::string("k_jk_stored_tma launch: ") + cudaGetErrorString(e));
            if (dK) {
                k_kslot_reduce<<<grid_for(ctx, (int64_t)nd * nn, 256, 8), 256, 0, ctx->stream>>>(Kslot, Krow, dK + d0 * nn, nd, n, grid, kslots);
                ctx->launches++;
                CK(cudaGetLastError());
            }
        }
        CK(cudaEventRecord(ctx->ev[2][1], ctx->stream));
        return TUNA_OK;
    }
    // ---- simple variant (any n) ----
    const int r = std::max(1, 256 / n);
    const int threads = (n * r + 31) / 32 * 32;
    const int lch = 4;
    const int nchunk = (n + lch - 1) / lch;
    const int nwarp = (threads + 31) / 32;
    const size_t need_kpart = (size_t)std::min(nD, 4) * n * nchunk * n;
    if (dK) GROW(ctx->d_Kpart, need_kpart);
    CK(cudaEventRecord(ctx->ev[2][0], ctx->stream));
    for (int d0 = 0; d0 < nD; d0 += 4) {
        const int nd = std::min(4, nD - d0);
        const size_t smem = ((size_t)nd * lch * nwarp + (size_t)nd * r * n) * sizeof(double);
        dim3 grid(nchunk, n);
        const double* P = dP + d0 * nn;
        double* J = dJ ? dJ + d0 * nn : nullptr;
        double* Kp = dK ? ctx->d_Kpart.get() : nullptr;
        switch (nd) {
            case 1: k_jk_stored<1><<<grid, threads, smem, ctx->stream>>>(ctx->d_eri_sph, P, J, Kp, n, r, lch, nchunk); break;
            case 2: k_jk_stored<2><<<grid, threads, smem, ctx->stream>>>(ctx->d_eri_sph, P, J, Kp, n, r, lch, nchunk); break;
            case 3: k_jk_stored<3><<<grid, threads, smem, ctx->stream>>>(ctx->d_eri_sph, P, J, Kp, n, r, lch, nchunk); break;
            default: k_jk_stored<4><<<grid, threads, smem, ctx->stream>>>(ctx->d_eri_sph, P, J, Kp, n, r, lch, nchunk); break;
        }
        ctx->launches++;
        CK(cudaGetLastError());
        if (dK) {
            k_kpart_reduce<<<grid_for(ctx, (int64_t)nd * nn, 256, 8), 256, 0, ctx->stream>>>(ctx->d_Kpart, dK + d0 * nn, nd, n, nchunk);
            ctx->launches++;
            CK(cudaGetLastError());
        }
    }
    CK(cudaEventRecord(ctx->ev[2][1], ctx->stream));
    return TUNA_OK;
} TUNA_CATCH

extern "C" {

int tuna_jk_stored(tuna_ctx* ctx, int nD, const double* P, double* J, double* K) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (!ctx->d_eri_sph || ctx->n_stored == 0) FAIL(TUNA_ERR_STATE, "tuna_jk_stored: no stored tensor resident");
    if (nD <= 0 || !P) FAIL(TUNA_ERR_ARG, "tuna_jk_stored: bad arguments");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n_stored;
    int rc;
    if ((rc = ensure_mats(ctx, nD, n, 0))) return rc;
    const size_t bytes = (size_t)nD * n * n * sizeof(double);
    double* hP = ctx->h_pin;
    double* hJ = hP + (size_t)nD * n * n;
    double* hK = hJ + (size_t)nD * n * n;
    std::memcpy(hP, P, bytes);
    CK(cudaMemcpyAsync(ctx->d_P, hP, bytes, cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = tuna_jk_stored_dev(ctx, nD, ctx->d_P, J ? ctx->d_J.get() : nullptr, K ? ctx->d_K.get() : nullptr))) return rc;
    if (J) CK(cudaMemcpyAsync(hJ, ctx->d_J, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (K) CK(cudaMemcpyAsync(hK, ctx->d_K, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (J) std::memcpy(J, hJ, bytes);
    if (K) std::memcpy(K, hK, bytes);
    return TUNA_OK;
} TUNA_CATCH

int tuna_set_shard(tuna_ctx* ctx, int rank, int nranks) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (nranks < 1 || rank < 0 || rank >= nranks) FAIL(TUNA_ERR_ARG, "tuna_set_shard: bad rank / nranks");
    CK(cudaSetDevice(ctx->device));
    drop_store(ctx);            // the store holds the rows of this rank's units only
    ctx->shard_rank = rank; ctx->shard_n = nranks;
    return TUNA_OK;
} TUNA_CATCH

int tuna_set_integral_store(tuna_ctx* ctx, int64_t budget_bytes) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (budget_bytes < 0) FAIL(TUNA_ERR_ARG, "tuna_set_integral_store: negative budget");
    CK(cudaSetDevice(ctx->device));
    if (budget_bytes != ctx->store_budget) drop_store(ctx);
    ctx->store_budget = budget_bytes;
    return TUNA_OK;
} TUNA_CATCH

int tuna_integral_store_info(const tuna_ctx* ctx, int64_t info[4]) {
    if (!ctx || !info) return TUNA_ERR_ARG;
    int64_t items = 0;
    for (const auto& e : ctx->store) if (e.filled) items += e.items;
    info[0] = items > 0 ? (int64_t)(ctx->d_store.capacity() * sizeof(double)) : 0;
    info[1] = items;
    info[2] = ctx->store_items_last;
    info[3] = ctx->store_replays;
    return TUNA_OK;
}

}  // extern "C" (internal helpers follow)

// ------------------------------------------------------------------------------------------------
// AO -> MO / spin-orbital transformation of the dense tensor (tuna_ci.py:143-255); kernel in mo_transform.cuh
// ------------------------------------------------------------------------------------------------
// Spin-blocked tensor of TUNA/tuna_ci.py:564, built on the device from the resident tensor E (dimension n):
//   G = np.kron(np.eye(2), np.kron(np.eye(2), E).T)  =>  G[I][J][K][L] = [I/n == J/n] [K/n == L/n] E[L%n][K%n][J%n][I%n]   (dimension 2n)
// (NumPy's kron pads eye(2) to four axes, so each kron spin-blocks the LAST two axes; the .T in between reverses all four.)
__global__ void __launch_bounds__(256) k_spin_block(const double* __restrict__ E, double* __restrict__ G, int n) {
    const int n2 = 2 * n;
    const size_t IJ = blockIdx.x;                       // one (I, J) plane per CTA
    const int I = (int)(IJ / n2), J = (int)(IJ % n2);
    double* g = G + IJ * (size_t)n2 * n2;
    const bool on = (I / n) == (J / n);
    const int i = I % n, j = J % n;
    for (int kl = threadIdx.x; kl < n2 * n2; kl += blockDim.x) {
        const int K = kl / n2, L = kl - K * n2;
        double v = 0.0;
        if (on && (K / n) == (L / n)) v = E[(((size_t)(L % n) * n + (K % n)) * n + j) * n + i];
        g[kl] = v;
    }
}

static int mo_transform_core(tuna_ctx* ctx, int n, const double* dT, int n1, const double* dC1, int n2, const double* dC2, int so_layout,
                             double* d_out) {
    const size_t N = (size_t)n, N1 = (size_t)n1, N2 = (size_t)n2;
    const size_t s1 = N1 * N * N * N, s2 = N1 * N1 * N * N, s3 = N2 * N1 * N1 * N;
    const size_t need[2] = {std::max(s1, s3), s2};
    for (int b = 0; b < 2; ++b)
        if (ctx->d_mo_ws[b].capacity() < need[b]) {
            CK(cudaStreamSynchronize(ctx->stream));
            GROW(ctx->d_mo_ws[b], need[b]);
        }
    double* A = ctx->d_mo_ws[0];
    double* B = ctx->d_mo_ws[1];
    CK(cudaEventRecord(ctx->ev[4][0], ctx->stream));
    CK(axis_gemm(ctx->stream, dT, dC1, A, (long long)(N * N * N), n, n1, 0, 0, 0, 0));          // (m k n l) -> (s m k n)
    CK(axis_gemm(ctx->stream, A, dC1, B, (long long)(N1 * N * N), n, n1, 0, 0, 0, 0));          //           -> (q s m k)
    CK(axis_gemm(ctx->stream, B, dC2, A, (long long)(N1 * N1 * N), n, n2, 0, 0, 0, 0));         //           -> (r q s m)
    CK(axis_gemm(ctx->stream, A, dC2, d_out, (long long)(N2 * N1 * N1), n, n2, so_layout ? 1 : 0, n2, n1, n1));   // -> (p r q s) | (p q r s)
    CK(cudaEventRecord(ctx->ev[4][1], ctx->stream));
    ctx->launches += 4;
    return TUNA_OK;
}

extern "C" {

int tuna_eri_transform_dev(tuna_ctx* ctx, int n, const double* dT, int n1, const double* dC1, int n2, const double* dC2, int so_layout,
                           double* d_out) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (n <= 0 || n1 <= 0 || n2 <= 0 || !dC1 || !dC2 || !d_out) FAIL(TUNA_ERR_ARG, "tuna_eri_transform: bad arguments");
    CK(cudaSetDevice(ctx->device));
    if (!dT) {
        if (!ctx->d_eri_sph || ctx->n_stored != n) FAIL(TUNA_ERR_STATE, "tuna_eri_transform: no stored tensor of that dimension is resident");
        dT = ctx->d_eri_sph;
    }
    return mo_transform_core(ctx, n, dT, n1, dC1, n2, dC2, so_layout, d_out);
} TUNA_CATCH

int tuna_eri_transform(tuna_ctx* ctx, int n, const double* eri_host, int n1, const double* C1, int n2, const double* C2, int so_layout,
                       double* out_host) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (n <= 0 || n1 <= 0 || n2 <= 0 || !C1 || !C2 || !out_host) FAIL(TUNA_ERR_ARG, "tuna_eri_transform: bad arguments");
    CK(cudaSetDevice(ctx->device));
    const size_t n4 = (size_t)n * n * n * n, nout = (size_t)n1 * n1 * n2 * n2;
    if (!eri_host && (!ctx->d_eri_sph || ctx->n_stored != n))
        FAIL(TUNA_ERR_STATE, "tuna_eri_transform: no stored tensor of that dimension is resident and no host tensor was given");
    DevBuf<double> dT, dC, dOut;
    if (eri_host) GROW(dT, n4);
    GROW(dC, (size_t)n * (n1 + n2));
    GROW(dOut, nout);
    if (eri_host) CK(cudaMemcpyAsync(dT, eri_host, n4 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dC, C1, (size_t)n * n1 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dC + (size_t)n * n1, C2, (size_t)n * n2 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    if (int rc = mo_transform_core(ctx, n, eri_host ? dT : ctx->d_eri_sph, n1, dC, n2, dC + (size_t)n * n1, so_layout, dOut)) return rc;
    CK(cudaMemcpyAsync(out_host, dOut, nout * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TUNA_OK;
} TUNA_CATCH

int tuna_eri_transform_spin_blocked(tuna_ctx* ctx, int n1, const double* C1, int n2, const double* C2, int so_layout, double* out_host) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (n1 <= 0 || n2 <= 0 || !C1 || !C2 || !out_host) FAIL(TUNA_ERR_ARG, "tuna_eri_transform_spin_blocked: bad arguments");
    if (!ctx->d_eri_sph || ctx->n_stored <= 0) FAIL(TUNA_ERR_STATE, "tuna_eri_transform_spin_blocked: no stored tensor is resident");
    CK(cudaSetDevice(ctx->device));
    const int n = ctx->n_stored, N = 2 * n;
    const size_t N4 = (size_t)N * N * N * N, nout = (size_t)n1 * n1 * n2 * n2;
    DevBuf<double> dG, dC, dOut;
    GROW(dG, N4);
    GROW(dC, (size_t)N * (n1 + n2));
    GROW(dOut, nout);
    CK(cudaMemcpyAsync(dC, C1, (size_t)N * n1 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(dC + (size_t)N * n1, C2, (size_t)N * n2 * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    k_spin_block<<<(unsigned)((size_t)N * N), 256, 0, ctx->stream>>>(ctx->d_eri_sph, dG, n);
    ctx->launches++;
    if (int rc = mo_transform_core(ctx, N, dG, n1, dC, n2, dC + (size_t)N * n1, so_layout, dOut)) return rc;
    CK(cudaMemcpyAsync(out_host, dOut, nout * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TUNA_OK;
} TUNA_CATCH

}  // extern "C"

// ------------------------------------------------------------------------------------------------
// One-electron integrals (SURVEY.md 8f-3): overlap, kinetic, nuclear attraction, dipole, diagonal quadrupole
// (tuna_integral.pyx:282-445) and the cross-basis overlap (:626-778); math in oneel_core.cuh
// ------------------------------------------------------------------------------------------------
struct BasisDev {       // kernel argument: a view of a BasisBuf
    int n = 0;
    double* oz = nullptr; int* lmn = nullptr; int* nprim = nullptr; int64_t* off = nullptr; double* exps = nullptr; double* ceff = nullptr;
};

struct BasisBuf {
    int n = 0;
    DevBuf<double> oz; DevBuf<int> lmn, nprim; DevBuf<int64_t> off; DevBuf<double> exps, ceff;
    BasisDev view() const { return BasisDev{n, oz, lmn, nprim, off, exps, ceff}; }
};

static int basis_dev_upload(tuna_ctx* ctx, BasisBuf& B, int n, const double* oz, const int32_t* lmn, const int32_t* nprim, const int64_t* off,
                            const double* exps, const double* ceff) {
    int64_t tot = 0;
    for (int i = 0; i < n; ++i) {
        if (nprim[i] <= 0) FAIL(TUNA_ERR_ARG, "basis function without primitives");
        for (int c = 0; c < 3; ++c)
            if (lmn[3 * i + c] < 0 || lmn[3 * i] + lmn[3 * i + 1] + lmn[3 * i + 2] > OE_LMAX) FAIL(TUNA_ERR_ARG, "angular momentum outside 0..5 (only up to H functions, tuna_molecule.py:612-618)");
        tot = std::max<int64_t>(tot, off[i] + nprim[i]);
    }
    B.n = n;
    GROW(B.oz, (size_t)n);
    GROW(B.lmn, (size_t)3 * n);
    GROW(B.nprim, (size_t)n);
    GROW(B.off, (size_t)n);
    GROW(B.exps, (size_t)tot);
    GROW(B.ceff, (size_t)tot);
    CK(cudaMemcpyAsync(B.oz, oz, (size_t)n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(B.lmn, lmn, (size_t)3 * n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(B.nprim, nprim, (size_t)n * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(B.off, off, (size_t)n * sizeof(int64_t), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(B.exps, exps, (size_t)tot * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaMemcpyAsync(B.ceff, ceff, (size_t)tot * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    return TUNA_OK;
}

// One thread per AO pair i >= j; out = [S | T | V | D(3) | Q(3)], nine n x n matrices, both triangles written.
__global__ void __launch_bounds__(128) k_one_electron(BasisDev B, int natoms, const double* __restrict__ atoms /* z[natoms] | charge[natoms] | origin[3] */,
                                                      const double* __restrict__ boys, double* __restrict__ out) {
    const long long n = B.n, idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= n * n) return;
    const int i = (int)(idx / n), j = (int)(idx % n);
    if (j > i) return;
    const OneElPair o = one_electron_pair(B.lmn + 3 * i, B.oz[i], B.nprim[i], B.exps + B.off[i], B.ceff + B.off[i], B.lmn + 3 * j, B.oz[j], B.nprim[j],
                                          B.exps + B.off[j], B.ceff + B.off[j], natoms, atoms, atoms + natoms, atoms + 2 * natoms, boys);
    const size_t nn = (size_t)n * n, ij = (size_t)i * n + j, ji = (size_t)j * n + i;
    out[ij] = o.s; out[ji] = o.s;
    out[nn + ij] = o.t; out[nn + ji] = o.t;
    out[2 * nn + ij] = o.v; out[2 * nn + ji] = o.v;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        out[(3 + c) * nn + ij] = o.d[c]; out[(3 + c) * nn + ji] = o.d[c];
        out[(6 + c) * nn + ij] = o.q[c]; out[(6 + c) * nn + ji] = o.q[c];
    }
}

__global__ void __launch_bounds__(128) k_cross_overlap(BasisDev A, BasisDev B, double* __restrict__ out) {
    const long long n2 = B.n, idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)A.n * n2) return;
    const int i = (int)(idx / n2), j = (int)(idx % n2);
    out[idx] = overlap_pair(A.lmn + 3 * i, A.oz[i], A.nprim[i], A.exps + A.off[i], A.ceff + A.off[i], B.lmn + 3 * j, B.oz[j], B.nprim[j], B.exps + B.off[j],
                            B.ceff + B.off[j]);
}

extern "C" {

int tuna_one_electron(tuna_ctx* ctx, int n_atoms, const double* atom_z, const double* atom_charge, const double* dipole_origin, double* S, double* T,
                      double* V, double* D, double* Q) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (ctx->ncart == 0) FAIL(TUNA_ERR_STATE, "tuna_one_electron: call tuna_set_basis first");
    if (n_atoms <= 0 || !atom_z || !atom_charge || !dipole_origin || !S || !T || !V || !D || !Q) FAIL(TUNA_ERR_ARG, "tuna_one_electron: bad arguments");
    CK(cudaSetDevice(ctx->device));
    const HostBasis& H = ctx->hb;
    const int n = ctx->ncart;
    const size_t nn = (size_t)n * n;
    std::vector<int32_t> np32(H.nprim.begin(), H.nprim.end()), lmn32(H.lmn.begin(), H.lmn.end());
    std::vector<double> at((size_t)2 * n_atoms + 3);
    for (int a = 0; a < n_atoms; ++a) { at[a] = atom_z[a]; at[n_atoms + a] = atom_charge[a]; }
    for (int c = 0; c < 3; ++c) at[2 * n_atoms + c] = dipole_origin[c];
    BasisBuf B;
    DevBuf<double> d_at, d_out;
    if (int rc = basis_dev_upload(ctx, B, n, H.oz.data(), lmn32.data(), np32.data(), H.off.data(), H.exps.data(), H.ceff.data())) return rc;
    GROW(d_at, at.size());
    GROW(d_out, 9 * nn);
    CK(cudaMemcpyAsync(d_at, at.data(), at.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaEventRecord(ctx->ev[5][0], ctx->stream));
    k_one_electron<<<(unsigned)((nn + 127) / 128), 128, 0, ctx->stream>>>(B.view(), n_atoms, d_at, ctx->d_boys, d_out);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaEventRecord(ctx->ev[5][1], ctx->stream));
    // straight into the caller's buffers (page-locked when they come from the Python layer): no staging vector, no second copy
    double* dst[5] = {S, T, V, D, Q};
    const size_t cnt[5] = {nn, nn, nn, 3 * nn, 3 * nn};
    size_t off = 0;
    for (int k = 0; k < 5; ++k) {
        CK(cudaMemcpyAsync(dst[k], d_out + off, cnt[k] * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        off += cnt[k];
    }
    CK(cudaStreamSynchronize(ctx->stream));
    return TUNA_OK;
} TUNA_CATCH

int tuna_cross_overlap(tuna_ctx* ctx, int n1, const double* oz1, const int32_t* lmn1, const int32_t* nprim1, const int64_t* off1, const double* exps1,
                       const double* ceff1, int n2, const double* oz2, const int32_t* lmn2, const int32_t* nprim2, const int64_t* off2,
                       const double* exps2, const double* ceff2, double* S12) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (n1 <= 0 || n2 <= 0 || !oz1 || !lmn1 || !nprim1 || !off1 || !exps1 || !ceff1 || !oz2 || !lmn2 || !nprim2 || !off2 || !exps2 || !ceff2 || !S12)
        FAIL(TUNA_ERR_ARG, "tuna_cross_overlap: bad arguments");
    CK(cudaSetDevice(ctx->device));
    BasisBuf A, B;
    DevBuf<double> d_out;
    const size_t count = (size_t)n1 * n2;
    int rc;
    if ((rc = basis_dev_upload(ctx, A, n1, oz1, lmn1, nprim1, off1, exps1, ceff1))) return rc;
    if ((rc = basis_dev_upload(ctx, B, n2, oz2, lmn2, nprim2, off2, exps2, ceff2))) return rc;
    GROW(d_out, count);
    k_cross_overlap<<<(unsigned)((count + 127) / 128), 128, 0, ctx->stream>>>(A.view(), B.view(), d_out);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(S12, d_out, count * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    return TUNA_OK;
} TUNA_CATCH

}  // extern "C"

// Shell-pair data of the shell-quartet engine (built once per geometry).
static int ensure_shell_pairs(tuna_ctx* ctx) {
    int rc;
    if (!ctx->shell_ready) {
        if ((rc = ensure_schwarz(ctx))) return rc;
        std::vector<double> q((size_t)ctx->pt.npair);
        CK(cudaMemcpyAsync(q.data(), ctx->d_Q, q.size() * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ShellSystem& S = ctx->ss;
        try {
            build_shell_pairs(S, ctx->stab, ctx->pt, q, ctx->ncart);
        } catch (const std::bad_alloc&) { FAIL(TUNA_ERR_NOMEM, "host allocation failed while building shell pairs"); }
        const size_t np = S.pairA.size();
        GROW(ctx->d_pairA, np);
        GROW(ctx->d_pairB, np);
        GROW(ctx->d_pair_rec, np);
        GROW(ctx->d_pairQ, np);
        GROW(ctx->d_rec, S.rec.size());
        GROW(ctx->d_sh_ao, S.sh_ao.size());
        GROW(ctx->d_finv, (size_t)ctx->ncart);
        GROW(ctx->d_fnorm, (size_t)ctx->ncart);
        GROW(ctx->d_eval, (size_t)1);
        std::vector<int> lists;
        ctx->class_list_off.clear();
        for (auto& c : S.classes) { ctx->class_list_off.push_back(lists.size()); lists.insert(lists.end(), c.pairs.begin(), c.pairs.end()); }
        GROW(ctx->d_class_lists, lists.size());
        std::vector<double> finv(ctx->ncart);
        for (int i = 0; i < ctx->ncart; ++i) finv[i] = 1.0 / S.fnorm[i];
        CK(cudaMemcpyAsync(ctx->d_pairA, S.pairA.data(), np * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_pairB, S.pairB.data(), np * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_pair_rec, S.pair_rec.data(), np * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_pairQ, S.pairQ.data(), np * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_rec, S.rec.data(), S.rec.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_sh_ao, S.sh_ao.data(), S.sh_ao.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_class_lists, lists.data(), lists.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_finv, finv.data(), finv.size() * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(ctx->d_fnorm, S.fnorm.data(), (size_t)ctx->ncart * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->shell_ready = true;
    }
    return TUNA_OK;
}

// ------------------------------------------------------------------------------------------------------------------------------
// generation-4 engine: per-class tables, job list, launches
// ------------------------------------------------------------------------------------------------------------------------------
constexpr int SHELL4_SMEM_DOUBLES = 27000;       // 211 KB of the 227 KB a CTA may use (tables and headers come on top)

static int shell4_slice_doubles(const Class4Host& C, int nD) {
    Shell4Job Jt;
    Jt.La = C.La; Jt.Lb = C.Lb; Jt.Lc = C.Lc; Jt.Ld = C.Ld;
    Jt.ct.ssize = C.ssize; Jt.ct.itmax = C.itmax; Jt.ct.zrow = C.zrow; Jt.ct.nstage = C.nstage; Jt.ct.nwork = C.nwork;
    Jt.ct.nout_sm = C.nterm2 > 0 ? 0 : C.nwork;
    shell4_job_layout(Jt, nD);
    return Jt.total + (C.tab_words + 1) / 2 + 16;
}

static int get_class4_tables(tuna_ctx* ctx, int La, int Lb, int Lc, int Ld, int nD, tuna_ctx::ClassTab4Dev** out) {
    const int key = La | Lb << 4 | Lc << 8 | Ld << 12 | nD << 16;
    auto it = ctx->class_tabs4.find(key);
    if (it != ctx->class_tabs4.end()) { *out = &it->second; return TUNA_OK; }
    tuna_ctx::ClassTab4Dev E;         // cached only once its blob is uploaded and its view set
    {
        const char* eb = getenv("TUNA_B200_IT_BUDGET");
        const char* es = getenv("TUNA_B200_S_BUDGET");
        const char* etm = getenv("TUNA_B200_TERM_MAX");
        int itb = eb ? atoi(eb) : S4_IT_BUDGET, sb = es ? atoi(es) : S4_S_BUDGET;
        const bool fill = nD == 0;                 // the fill job set: explicit (slot, components) lists, separable tables, no densities
        const int tmax = fill ? 0 : etm ? atoi(etm) : S4_TERM_MAX;
        build_class4_tables(ctx->stab, La, Lb, Lc, Ld, E.host, itb, sb, tmax, fill);
        // a slice that does not fit one CTA is re-cut into more chunks; a slice between half and all of an SM's shared memory is
        // re-cut so that two CTAs fit (phases 0-2 then run once per chunk)
        const int tier2 = (225 * 1024 / 2 - 1024 - 64) / 8;
        for (int pass = 0; pass < 6; ++pass) {
            const int t0 = shell4_slice_doubles(E.host, nD);
            const bool too_big = t0 > SHELL4_SMEM_DOUBLES;
            const char* et = getenv("TUNA_B200_TIER2");
            const bool tier = t0 > tier2 && !(et && atoi(et) == 0) && pass < 3;
            if (!too_big && !tier) break;
            const int nch = (int)E.host.chunk_row0.size() - 1;
            Class4Host trial;
            bool found = false;
            for (int want = nch + 1; want <= nch + 3 && !found; ++want) {
                build_class4_tables(ctx->stab, La, Lb, Lc, Ld, trial, std::max(64, E.host.nint / want + E.host.nint / (8 * want)), 65000, tmax, fill);
                if ((int)trial.chunk_row0.size() - 1 > nch && (shell4_slice_doubles(trial, nD) <= (too_big ? SHELL4_SMEM_DOUBLES : tier2))) found = true;
            }
            if (found) { E.host = trial; if (!too_big) break; }
            else if (!too_big) break;
            else if (pass == 5) FAIL(TUNA_ERR_STATE, "shell engine: class does not fit shared memory");
            else { build_class4_tables(ctx->stab, La, Lb, Lc, Ld, trial, std::max(64, E.host.itmax / 2), std::max(64, E.host.ssize / 2), tmax, fill); E.host = trial; }
        }
    }
    const Class4Host& C = E.host;
    size_t total = 0;
    auto reserve = [&](size_t bytes) { size_t o = total; total += (bytes + 15) & ~(size_t)15; return o; };
    struct Piece { const void* src; size_t bytes, off; };
    std::vector<Piece> pieces;
    auto add = [&](const void* src, size_t bytes) { pieces.push_back({src, bytes, reserve(bytes)}); return pieces.back().off; };
    const size_t o_rt = add(C.t_rt.data(), C.t_rt.size() * 4), o_xy = add(C.t_xy.data(), C.t_xy.size() * 4), o_u = add(C.t_u.data(), C.t_u.size() * 4);
    const size_t o_s = add(C.t_s.data(), C.t_s.size() * 4), o_s0 = add(C.chunk_s0.data(), C.chunk_s0.size() * 4), o_p4 = add(C.p4.data(), C.p4.size() * 4);
    const size_t o_t0 = add(C.chunk_t0.data(), C.chunk_t0.size() * 4), o_ni = add(C.chunk_ni.data(), C.chunk_ni.size() * 4);
    const size_t o_pmap = add(C.pmap.data(), C.pmap.size() * 2), o_omap = add(C.omap.data(), C.omap.size() * 2);
    const size_t o_jp = add(C.jst_ptr.data(), C.jst_ptr.size() * 4), o_jl = add(C.jst_list.data(), C.jst_list.size() * 2), o_jf = add(C.jflush.data(), C.jflush.size() * 4);
    const size_t o_acc = add(C.acc.data(), C.nterm2 > 0 ? 0 : C.acc.size() * 4);      // (unused in term mode)
    const size_t o_tabs = add(C.tabs.data(), C.tabs.size() * 4);
    const size_t o_tm = add(C.terms.data(), C.terms.size() * 4), o_tp = add(C.tptr.data(), C.tptr.size() * 4);
    const size_t o_wf = add(C.wfl.data(), C.wfl.size() * 4), o_wl = add(C.wlist.data(), C.wlist.size() * 2);
    const size_t o_fl = add(C.fill.data(), C.fill.size() * 4), o_f0 = add(C.chunk_f0.data(), C.chunk_f0.size() * 4), o_fp = add(C.fperm.data(), C.fperm.size() * 4);
    const size_t o_cn = add(C.canon.data(), C.canon.size() * 4), o_c0 = add(C.chunk_c0.data(), C.chunk_c0.size() * 4);
    std::vector<unsigned char> host(total, 0);
    for (const Piece& p : pieces) if (p.bytes) std::memcpy(host.data() + p.off, p.src, p.bytes);
    GROW(E.blob, total);
    CK(cudaMemcpyAsync(E.blob, host.data(), total, cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    Class4Dev& V = E.view;
    V = class4_view(C, HostPtrOf());          // scalars; the pointers are replaced by device addresses below
    V.t_rt = (const unsigned*)(E.blob + o_rt); V.t_xy = (const unsigned*)(E.blob + o_xy); V.t_u = (const unsigned*)(E.blob + o_u);
    V.t_s = (const unsigned*)(E.blob + o_s); V.chunk_s0 = (const int*)(E.blob + o_s0); V.p4 = (const unsigned*)(E.blob + o_p4);
    V.chunk_t0 = (const int*)(E.blob + o_t0); V.chunk_ni = (const int*)(E.blob + o_ni); V.tabs = (const unsigned*)(E.blob + o_tabs);
    V.acc = (const unsigned*)(E.blob + o_acc); V.pmap = (const unsigned short*)(E.blob + o_pmap); V.omap = (const unsigned short*)(E.blob + o_omap);
    V.jst_ptr = (const unsigned*)(E.blob + o_jp); V.jst_list = (const unsigned short*)(E.blob + o_jl); V.jflush = (const unsigned*)(E.blob + o_jf);
    V.terms = (const unsigned*)(E.blob + o_tm); V.tptr = (const unsigned*)(E.blob + o_tp);
    V.wfl = (const unsigned*)(E.blob + o_wf); V.wlist = (const unsigned short*)(E.blob + o_wl);
    V.fill = (const unsigned*)(E.blob + o_fl); V.chunk_f0 = (const int*)(E.blob + o_f0); V.fperm = (const unsigned*)(E.blob + o_fp);
    V.canon = (const unsigned*)(E.blob + o_cn); V.chunk_c0 = (const int*)(E.blob + o_c0);
    *out = &ctx->class_tabs4.emplace(key, std::move(E)).first->second;
    return TUNA_OK;
}

// Register budget of a job's own k_shell4_one launch.  A G = 256, NB <= 2 class whose shared-memory footprint already limits the SM to
// two 256-thread CTAs gets the 128-register build (no spills, more loads in flight in the unrolled digestion); TUNA_B200_REG_TIER=0
// forces the default build.  Grouped jobs (k_shell4_multi) always use the default build.
static int shell4_one_regs(const tuna_ctx::Job4Host& jh) {
    static const bool tiers = !(getenv("TUNA_B200_REG_TIER") && atoi(getenv("TUNA_B200_REG_TIER")) == 0);
    const size_t by_smem = std::max<size_t>(1, (size_t)(228 * 1024) / (jh.smem + 1024));
    return tiers && jh.G == 256 && jh.nb <= 2 && by_smem * jh.threads * 128 <= 65536 ? 128 : TUNA_SHELL4_REGS;
}

// ---- integral store (semi-direct J/K) --------------------------------------------------------------------------------------------
// Estimated phase 0-4 work of one work item (arbitrary units, one per FMA-sized step): the Boys values of phase 0, the entries of phases
// 1-3 and the assembly FMAs of the phase-4 tiles, per primitive quartet, times the primitive quartets of the item.
static double store_cost_per_item(const Class4Host& C, const Shell4Job& J) {
    const int Ltot = C.La + C.Lb + C.Lc + C.Ld;
    double w = 40.0 * (Ltot + 1) + 4.0 * (C.t_rt.size() + C.t_xy.size() + C.t_u.size() / 2 + C.t_s.size() / 2);
    for (size_t t = 0; t < C.p4.size(); t += 4) {
        const unsigned w2 = C.p4[t + 2];
        const int nx = (int)((w2 >> 4) & 15) - (int)(w2 & 15) + 1, ny = (w2 >> 12) & 15;
        w += nx * (2.0 * ny + 2.0);
    }
    return w * (double)J.clen * (double)J.klen;
}

// This rank's share of job jh: the units its launch deals to it (shell4_store_share, shell4_store_row).
static StoreShare store_share(const tuna_ctx* ctx, const tuna_ctx::Job4Host& jh) {
    return shell4_store_share(jh.job.nitems * jh.job.psplit, jh.job.chunk, jh.unit0, ctx->shard_rank, ctx->shard_n);
}

static void drop_store(tuna_ctx* ctx) {
    if (ctx->d_store) cudaStreamSynchronize(ctx->stream);      // no build in flight reads the rows any more
    ctx->store.clear();
    ctx->d_store.reset();
    ctx->store_planned = false;
}

// Plans the store from the current job set: whole jobs by decreasing cost per byte while they fit the budget, the budget clamped to the
// device's free memory less headroom for the build's own buffers.  One allocation; if it fails the store stays empty (the builds run
// direct) until the budget is set again.
static void plan_store(tuna_ctx* ctx) {
    ctx->store_planned = true;
    ctx->store.clear();
    const auto& jobs = ctx->jobsets4[ctx->cur_jobset4].jobs;
    size_t free_b = 0, total_b = 0;
    if (cudaMemGetInfo(&free_b, &total_b) != cudaSuccess) { cudaGetLastError(); return; }
    const size_t headroom = std::max<size_t>((size_t)2 << 30, total_b / 16);
    const long long budget = std::min<long long>(ctx->store_budget, free_b > headroom ? (long long)(free_b - headroom) : 0);
    std::vector<int> order(jobs.size());
    for (size_t j = 0; j < jobs.size(); ++j) order[j] = (int)j;
    std::stable_sort(order.begin(), order.end(), [&](int x, int y) { return jobs[x].cost_per_byte > jobs[y].cost_per_byte; });
    long long used = 0;      // doubles
    for (int j : order) {
        const tuna_ctx::Job4Host& jh = jobs[j];
        const StoreShare sh = store_share(ctx, jh);
        const long long need = sh.rows * jh.job.ct.nint;
        if (need == 0 || (used + need) * 8 > budget) continue;
        ctx->store.push_back({jh.cb, jh.ck, jh.job.psplit, jh.job.chunk, jh.job.ct.nint, jh.list_sum, jh.unit0, used, sh.items, false});
        used += need;
    }
    if (used == 0) return;
    std::string err;
    if (ctx->d_store.grow((size_t)used, err) != TUNA_OK) ctx->store.clear();      // optional memory: run direct, report nothing
}

// Mode of job jh in this build, and its first row.  A stored job whose kept quartet list or split differs from the stored one runs
// direct, and so does one whose unit size or flat unit offset (own launch or grouped, the group's other jobs) differs on a sharded
// context, where they decide which units, hence rows, the rank owns.  Such a job is not stored again.
static int store_mode_of(const tuna_ctx* ctx, const tuna_ctx::Job4Host& jh, long long* base) {
    for (const auto& e : ctx->store) {
        if (e.cb != jh.cb || e.ck != jh.ck) continue;
        if (e.list_sum != jh.list_sum || e.psplit != jh.job.psplit || e.nint != jh.job.ct.nint || (ctx->shard_n > 1 && (e.chunk != jh.job.chunk || e.unit0 != jh.unit0)))
            return S4_DIRECT;
        *base = e.base;
        return e.filled ? S4_REPLAY : S4_STORE;
    }
    return S4_DIRECT;
}

// Job list of the shell-quartet engine for threshold tau and nD densities.
static int ensure_shell4(tuna_ctx* ctx, double tau, int nD) {
    int rc;
    if ((rc = ensure_shell_pairs(ctx))) return rc;
    for (size_t i = 0; i < ctx->jobsets4.size(); ++i)
        if (ctx->jobsets4[i].tau == tau && ctx->jobsets4[i].nD == nD && ctx->jobsets4[i].shard_n == ctx->shard_n && ctx->jobsets4[i].dens_bound >= ctx->dens_bound) {
            ctx->cur_jobset4 = (int)i;
            return TUNA_OK;
        }
    ctx->cur_jobset4 = -1;
    if (ctx->jobsets4.size() >= 6) {
        CK(cudaStreamSynchronize(ctx->stream));
        ctx->jobsets4.erase(ctx->jobsets4.begin());
    }
    tuna_ctx::JobSet4 JS;         // cached only once complete: a failed build frees whatever it allocated
    JS.tau = tau; JS.nD = nD; JS.shard_n = ctx->shard_n; JS.dens_bound = ctx->dens_bound;
    std::vector<tuna_ctx::Job4Host>& jobs4 = JS.jobs;
    const ShellSystem& S = ctx->ss;
    const int ncls = (int)S.classes.size();
    std::vector<long long> all_prefix;
    std::vector<size_t> prefix_off;
    const bool fill = nD == 0;                  // dense-tensor fill: no densities, every work item writes a scratch row
    long long fill_run = 0;
    std::vector<std::pair<int, int>> job_cls;   // (bra class, ket class) of every job, in push order
    const char* env_div = getenv("TUNA_B200_G_DIV");
    const char* env_spl = getenv("TUNA_B200_SMEM_PER_LANE");
    const char* env_nb = getenv("TUNA_B200_NB");
    const char* env_nbmax = getenv("TUNA_B200_NB_BYTES");
    const double gdiv = env_div ? atof(env_div) : 8.0;
    const double smem_per_lane = env_spl ? atof(env_spl) : 256.0;
    const size_t nb_bytes = env_nbmax ? (size_t)atol(env_nbmax) : 100 * 1024;
    // static pre-screening uses the weakest density bound the device test can see (ADVICE r1: not a hard-coded 1e-3)
    for (int cb = 0; cb < ncls; ++cb)
        for (int ck = 0; ck <= cb; ++ck) {
            tuna_ctx::Job4Host jh;
            Shell4Job& J = jh.job;
            J.La = S.classes[cb].La; J.Lb = S.classes[cb].Lb; J.Lc = S.classes[ck].La; J.Ld = S.classes[ck].Lb;
            J.nppAB = S.classes[cb].npp; J.nppCD = S.classes[ck].npp;
            {   // at most ~psplit_target primitive quartets per work item (TUNA_B200_PSPLIT_TARGET, 0 = never split; TUNA_B200_KSPLIT=0: bra only)
                static const int target = getenv("TUNA_B200_PSPLIT_TARGET") ? atoi(getenv("TUNA_B200_PSPLIT_TARGET")) : 16;
                static const bool split_ket = !(getenv("TUNA_B200_KSPLIT") && atoi(getenv("TUNA_B200_KSPLIT")) == 0);
                shell4_split(J, target, split_ket);
            }
            { const char* dbg = getenv("TUNA_B200_DBG_SKIP"); J.dbg_skip = dbg ? atoi(dbg) : 0; }
            J.fill_scratch = nullptr; J.fill_base = 0; J.fill_pairs = nullptr;
            std::vector<long long> prefix;
            J.nitems = build_item_prefix(S, cb, ck, tau / ctx->dens_bound, prefix);
            if (J.nitems == 0) continue;
            J.nbra = (int)S.classes[cb].pairs.size(); J.same_class = (cb == ck);
            J.bra_list = ctx->d_class_lists + ctx->class_list_off[cb];
            J.ket_list = ctx->d_class_lists + ctx->class_list_off[ck];
            prefix_off.push_back(all_prefix.size());
            all_prefix.insert(all_prefix.end(), prefix.begin(), prefix.end());
            tuna_ctx::ClassTab4Dev* ctd = nullptr;
            if ((rc = get_class4_tables(ctx, J.La, J.Lb, J.Lc, J.Ld, nD, &ctd))) return rc;
            J.ct = ctd->view;
            shell4_job_layout(J, nD);
            if (fill) { J.fill_base = fill_run; fill_run += J.nitems * J.psplit * J.ct.nfill; }
            jh.allowed = (double)ctd->host.allowed;
            for (int u = 0; u < 6; ++u) J.uniq[u] = ctd->host.uniq[u];
            jh.cb = cb; jh.ck = ck;
            jh.list_sum = checksum(prefix.data(), prefix.size() * sizeof(long long), (uint64_t)J.nitems);
            jh.cost_per_byte = store_cost_per_item(ctd->host, J) / (8.0 * ctd->host.nint);
            int nb = env_nb ? atoi(env_nb) : 2;
            if (nb != 1 && nb != 2 && nb != 4) nb = 2;
            while (nb > 1 && (size_t)nb * J.total * 8 > nb_bytes) nb >>= 1;
            int G = 1;
            while (G < 256 && G * gdiv < jh.allowed) G *= 2;
            while (G < 256 && (double)nb * J.total * 8.0 / G > smem_per_lane) G *= 2;
            while (G < 256 && (size_t)(G <= 32 ? 128 / G : 1) * nb * J.total * 8 > 190 * 1024) G *= 2;
            if (J.ct.nchunk > 1 && G < 64) G = 64;                 // the table reload of a multi-chunk class synchronises the whole CTA
            jh.G = G; jh.nb = nb;
            jh.threads = G <= 32 ? 128 : G;
            jh.gpc = jh.threads / G;
            {   // items per CTA work unit: enough units to spread over all CTA slots of all ranks eight times, at most 16 per group
                const size_t by_smem = std::max<size_t>(1, (size_t)(228 * 1024) / ((size_t)jh.gpc * nb * J.total * 8 + 2048));
                const long long slots = (long long)ctx->sm_count * (long long)std::min<size_t>(by_smem, 2048 / jh.threads) * ctx->shard_n;
                long long per = J.nitems * J.psplit / std::max<long long>(1, slots * 8 * jh.gpc);
                per = std::max<long long>(nb, std::min<long long>(per, 16));
                per = (per + nb - 1) / nb * nb;
                J.chunk = jh.gpc * (int)per;
            }
            const size_t slices = (size_t)jh.gpc * nb * J.total;
            J.tab_off = (int)((slices + 1) & ~(size_t)1);
            J.hdr_off = J.tab_off + (ctd->host.tab_words + 4 + 1) / 2;
            jh.smem = ((size_t)J.hdr_off + (size_t)J.chunk * sizeof(Quartet4) / 8 + 2) * sizeof(double);
            if (jh.smem > 226 * 1024) FAIL(TUNA_ERR_STATE, "shell engine: shared-memory layout exceeds 226 KB");
            jobs4.push_back(jh);
            job_cls.push_back({cb, ck});
        }
    GROW(JS.d_prefix, std::max<size_t>(all_prefix.size(), 1));
    CK(cudaMemcpyAsync(JS.d_prefix, all_prefix.data(), all_prefix.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    for (size_t j = 0; j < jobs4.size(); ++j) jobs4[j].job.item_prefix = JS.d_prefix + prefix_off[j];
    if (fill) {
        GROW(JS.d_scratch, (size_t)std::max<long long>(fill_run, 1));
        // (bra pair, ket pair) of every item, job after job in the order of all_prefix
        std::vector<int> fpairs;
        std::vector<size_t> fp_off;
        for (size_t j = 0; j < jobs4.size(); ++j) {
            const int cb = job_cls[j].first, ck = job_cls[j].second;
            const long long* pf = all_prefix.data() + prefix_off[j];
            fp_off.push_back(fpairs.size());
            for (size_t ib = 0; ib < S.classes[cb].pairs.size(); ++ib)
                for (long long k = 0; k < pf[ib + 1] - pf[ib]; ++k) { fpairs.push_back(S.classes[cb].pairs[ib]); fpairs.push_back(S.classes[ck].pairs[(size_t)k]); }
        }
        GROW(JS.d_fill_pairs, std::max<size_t>(fpairs.size(), 1));
        CK(cudaMemcpyAsync(JS.d_fill_pairs, fpairs.data(), fpairs.size() * sizeof(int), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        for (size_t j = 0; j < jobs4.size(); ++j) { jobs4[j].job.fill_scratch = JS.d_scratch; jobs4[j].job.fill_pairs = JS.d_fill_pairs + fp_off[j]; }
    }
    std::stable_sort(jobs4.begin(), jobs4.end(), [](const tuna_ctx::Job4Host& x, const tuna_ctx::Job4Host& y) {
        return x.allowed * (double)x.job.nitems > y.allowed * (double)y.job.nitems;
    });
    // light class jobs (two quartets per batch, little work) share one persistent launch per group size; the others get their own launch
    {
        // a job that cannot fill the GPU once with its own work units (TUNA_B200_OWN_LAUNCH_UNITS per SM and rank, default 2) is "light":
        // measured, the shared-memory descriptor of the grouped kernel costs ~25 % per quartet, so jobs with plenty of units keep their
        // own launch (even-tempered sweep), while the hundreds of tiny class jobs of a contracted basis collapse into a few launches
        // (N2/cc-pVTZ 231 -> 19 launches, 3.0 -> 1.5 ms per direct build)
        const char* et = getenv("TUNA_B200_OWN_LAUNCH_UNITS");
        const double per_sm = et ? atof(et) : 2.0;
        for (auto& jh : jobs4) {
            const double units = (double)((jh.job.nitems * jh.job.psplit + jh.job.chunk - 1) / jh.job.chunk);
            jh.own_launch = jh.nb != 2 || units >= per_sm * ctx->sm_count * ctx->shard_n;
        }
        for (int G = 256; G >= 1; G >>= 1) {
            std::vector<Shell4Job> js;
            std::vector<int> members;
            std::vector<long long> up(1, 0);
            size_t max_smem = 0;
            int threads = 128;
            for (size_t j = 0; j < jobs4.size(); ++j) {
                const auto& jh = jobs4[j];
                if (jh.own_launch || jh.G != G) continue;
                js.push_back(jh.job);
                members.push_back((int)j);
                up.push_back(up.back() + (jh.job.nitems * jh.job.psplit + jh.job.chunk - 1) / jh.job.chunk);
                max_smem = std::max(max_smem, jh.smem);
                threads = jh.threads;
            }
            if (js.size() < 2) { for (auto& jh : jobs4) if (!jh.own_launch && jh.G == G) jh.own_launch = true; continue; }
            for (size_t i = 0; i < members.size(); ++i) jobs4[members[i]].unit0 = up[i];      // ranks own the group's FLAT units
            tuna_ctx::Group4 g;
            g.G = G; g.threads = threads; g.njobs = (int)js.size(); g.nunits = up.back();
            g.job_off = (int)(((max_smem + 7) / 8 + 1) & ~(size_t)1);
            g.smem = (size_t)g.job_off * 8 + sizeof(Shell4Job) + 16;
            g.ctas_per_sm = (int)std::max<size_t>(1, std::min<size_t>(2048 / threads, (228 * 1024) / (g.smem + 1024)));
            GROW(g.d_jobs, js.size());
            GROW(g.d_unit_prefix, up.size());
            CK(cudaMemcpyAsync(g.d_jobs, js.data(), js.size() * sizeof(Shell4Job), cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaMemcpyAsync(g.d_unit_prefix, up.data(), up.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
            CK(cudaStreamSynchronize(ctx->stream));
            g.members = std::move(members);
            g.host_jobs = std::move(js);
            JS.groups.push_back(std::move(g));
        }
    }
    if (fill) {       // descriptors of ALL jobs and the prefix of their (shell quartet, fill entry) counts for the scatter pass
        std::vector<Shell4Job> js;
        std::vector<long long> pre(1, 0);
        for (const auto& jh : jobs4) {      // groups of whole shell quartets (k_fill_scatter)
            const long long nf = std::max(1, jh.job.ct.nfill), ipg = nf >= 256 ? 1 : 256 / nf;
            js.push_back(jh.job); pre.push_back(pre.back() + (jh.job.nitems + ipg - 1) / ipg);
        }
        JS.scatter_total = pre.back();
        GROW(JS.d_all_jobs, std::max<size_t>(js.size(), 1));
        GROW(JS.d_scatter_pre, pre.size());
        CK(cudaMemcpyAsync(JS.d_all_jobs, js.data(), js.size() * sizeof(Shell4Job), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaMemcpyAsync(JS.d_scatter_pre, pre.data(), pre.size() * sizeof(long long), cudaMemcpyHostToDevice, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
    }
    if (const char* dump = getenv("TUNA_B200_DUMP_JOBS")) {       // development aid: the job table in launch order
        if (FILE* f = fopen(dump, "w")) {
            // regs: register budget of the kernel build that runs the job; terms: 1 = term-list digestion, 0 = separable;
            // psplit / ksplit: work items per shell quartet and ket chunks among them
            fprintf(f, "idx,La,Lb,Lc,Ld,nppAB,nppCD,G,nb,threads,smem,total,nout,nint,itmax,nchunk,nitems,allowed,own,regs,terms,psplit,ksplit,nD\n");
            int idx = 0;
            for (const auto& jh : jobs4)
                fprintf(f, "%d,%d,%d,%d,%d,%d,%d,%d,%d,%d,%zu,%d,%d,%d,%d,%d,%lld,%.0f,%d,%d,%d,%d,%d,%d\n", idx++, jh.job.La, jh.job.Lb, jh.job.Lc, jh.job.Ld,
                        jh.job.nppAB, jh.job.nppCD, jh.G, jh.nb, jh.threads, jh.smem, jh.job.total, jh.job.ct.nwork, jh.job.ct.itmax, jh.job.ct.itmax,
                        jh.job.ct.nchunk, jh.job.nitems, jh.allowed, (int)jh.own_launch, jh.own_launch ? shell4_one_regs(jh) : TUNA_SHELL4_REGS,
                        (int)(jh.job.ct.nterm2 > 0), jh.job.psplit, jh.job.ksplit, nD);
            fclose(f);
        }
    }
    ctx->jobsets4.push_back(std::move(JS));
    ctx->cur_jobset4 = (int)ctx->jobsets4.size() - 1;
    return TUNA_OK;
}

template <int GG, int NB, int REGS, bool SEMI>
static cudaError_t launch_shell4_one_r(tuna_ctx* ctx, const tuna_ctx::Job4Host& jh, const ShellData& D, int nD, const double* Pf, const double* Psym,
                                       double* Jf, double* Kf, double tau, cudaStream_t stream, long long blocks) {
    if (cudaError_t e = opt_in_smem<k_shell4_one<GG, NB, REGS, SEMI>>(ctx); e != cudaSuccess) return e;
    k_shell4_one<GG, NB, REGS, SEMI><<<(int)blocks, jh.threads, jh.smem, stream>>>(jh.job, D, nD, Pf, Psym, Jf, Kf, ctx->ncart, tau, ctx->d_scalars, ctx->d_eval,
                                                                            ctx->shard_rank, ctx->shard_n);
    ctx->launches++;
    return cudaGetLastError();
}

template <int GG, int NB>
static cudaError_t launch_shell4_one(tuna_ctx* ctx, const tuna_ctx::Job4Host& jh, const ShellData& D, int nD, const double* Pf, const double* Psym,
                                     double* Jf, double* Kf, double tau, cudaStream_t stream) {
    const long long nunit = (jh.job.nitems * jh.job.psplit + jh.job.chunk - 1) / jh.job.chunk;
    long long blocks = (nunit - ctx->shard_rank + ctx->shard_n - 1) / ctx->shard_n;       // units owned by this rank
    if (blocks <= 0) return cudaSuccess;
    const size_t by_smem = std::max<size_t>(1, (size_t)(228 * 1024) / (jh.smem + 1024));
    const size_t by_thr = std::max<size_t>(1, 2048 / jh.threads);
    blocks = std::min<long long>(blocks, (long long)ctx->sm_count * (long long)std::min(by_smem, by_thr) * 2);
    const bool semi = jh.job.store_mode != S4_DIRECT;      // store pass or replay: the kernel variant with the integral-store paths
    if constexpr (GG == 256 && NB <= 2) {
        if (shell4_one_regs(jh) == 128)
            return semi ? launch_shell4_one_r<GG, NB, 128, true>(ctx, jh, D, nD, Pf, Psym, Jf, Kf, tau, stream, blocks)
                        : launch_shell4_one_r<GG, NB, 128, false>(ctx, jh, D, nD, Pf, Psym, Jf, Kf, tau, stream, blocks);
    }
    return semi ? launch_shell4_one_r<GG, NB, TUNA_SHELL4_REGS, true>(ctx, jh, D, nD, Pf, Psym, Jf, Kf, tau, stream, blocks)
                : launch_shell4_one_r<GG, NB, TUNA_SHELL4_REGS, false>(ctx, jh, D, nD, Pf, Psym, Jf, Kf, tau, stream, blocks);
}

template <int GG, bool SEMI>
static cudaError_t launch_shell4_multi(tuna_ctx* ctx, const tuna_ctx::Group4& g, const ShellData& D, int nD, const double* Pc, const double* Psym,
                                       double* Jc, double* Kc, double tau, cudaStream_t st, long long blocks) {
    if (cudaError_t e = opt_in_smem<k_shell4_multi<GG, 2, SEMI>>(ctx); e != cudaSuccess) return e;
    k_shell4_multi<GG, 2, SEMI><<<(int)blocks, g.threads, g.smem, st>>>(g.d_jobs, g.d_unit_prefix, g.njobs, g.job_off, D, nD, Pc, Psym, Jc, Kc, ctx->ncart,
                                                                     tau, ctx->d_scalars, ctx->d_eval, ctx->shard_rank, ctx->shard_n);
    return cudaGetLastError();
}

static int launch_shell4_jobs(tuna_ctx* ctx, int nD, const double* Pc, const double* Psym, double* Jc, double* Kc, double tau, long long fix_lo) {
    ShellData D;
    D.pairA = ctx->d_pairA; D.pairB = ctx->d_pairB; D.pair_rec = ctx->d_pair_rec; D.rec = ctx->d_rec; D.pairQ = ctx->d_pairQ;
    D.sh_ao = ctx->d_sh_ao; D.boys = ctx->d_boys; D.herm = ctx->d_herm;
    D.fix_lo = fix_lo;
    tuna_ctx::JobSet4& JS = ctx->jobsets4[ctx->cur_jobset4];
    // integral store: every job's mode in this build (direct / store pass / replay); the fill job set (nD = 0) never uses it
    const bool use_store = nD > 0 && ctx->store_budget > 0;
    if (use_store && !ctx->store_planned) plan_store(ctx);
    std::vector<int> modes(JS.jobs.size(), S4_DIRECT);
    std::vector<long long> bases(JS.jobs.size(), 0);
    if (use_store) {
        long long items_all = 0;
        for (size_t j = 0; j < JS.jobs.size(); ++j) {
            modes[j] = store_mode_of(ctx, JS.jobs[j], &bases[j]);
            items_all += store_share(ctx, JS.jobs[j]).items;
        }
        ctx->store_items_last = items_all;
    }
    auto with_store = [&](Shell4Job& J, size_t j) {
        J.store = modes[j] == S4_DIRECT ? nullptr : ctx->d_store.get();
        J.store_base = bases[j]; J.store_mode = modes[j]; J.store_nranks = ctx->shard_n;
        J.store_unit0 = JS.jobs[j].unit0; J.store_ubase = store_share(ctx, JS.jobs[j]).ubase;
    };
    for (auto& g : JS.groups) {          // grouped descriptors live on the device: re-upload when a job's store fields change
        bool changed = false;
        for (size_t i = 0; i < g.members.size(); ++i) {
            Shell4Job want = g.host_jobs[i];
            with_store(want, (size_t)g.members[i]);
            Shell4Job& have = g.host_jobs[i];
            if (want.store != have.store || want.store_base != have.store_base || want.store_mode != have.store_mode || want.store_nranks != have.store_nranks ||
                want.store_unit0 != have.store_unit0 || want.store_ubase != have.store_ubase) {
                have = want;
                changed = true;
            }
        }
        if (changed) CK(cudaMemcpyAsync(g.d_jobs, g.host_jobs.data(), g.host_jobs.size() * sizeof(Shell4Job), cudaMemcpyHostToDevice, ctx->stream));
    }
    CK(cudaEventRecord(ctx->ev_fork, ctx->stream));
    for (int a = 0; a < ctx->naux; ++a) CK(cudaStreamWaitEvent(ctx->aux[a], ctx->ev_fork, 0));
    int jn = 0;
    for (size_t j = 0; j < JS.jobs.size(); ++j) {
        if (!JS.jobs[j].own_launch) continue;
        tuna_ctx::Job4Host jh = JS.jobs[j];
        with_store(jh.job, j);
        cudaStream_t st = ctx->aux[jn++ % ctx->naux];
        cudaError_t e;
#define TUNA_ONE4(GV) (jh.nb == 4 ? launch_shell4_one<GV, 4>(ctx, jh, D, nD, Pc, Psym, Jc, Kc, tau, st) \
                       : jh.nb == 2 ? launch_shell4_one<GV, 2>(ctx, jh, D, nD, Pc, Psym, Jc, Kc, tau, st) \
                                    : launch_shell4_one<GV, 1>(ctx, jh, D, nD, Pc, Psym, Jc, Kc, tau, st))
        switch (jh.G) {
            case 1: e = TUNA_ONE4(1); break;
            case 2: e = TUNA_ONE4(2); break;
            case 4: e = TUNA_ONE4(4); break;
            case 8: e = TUNA_ONE4(8); break;
            case 16: e = TUNA_ONE4(16); break;
            case 32: e = TUNA_ONE4(32); break;
            case 64: e = TUNA_ONE4(64); break;
            case 128: e = TUNA_ONE4(128); break;
            default: e = TUNA_ONE4(256); break;
        }
#undef TUNA_ONE4
        if (e != cudaSuccess) FAIL(TUNA_ERR_CUDA, std::string("k_shell4_one launch: ") + cudaGetErrorString(e));
    }
    for (const auto& g : JS.groups) {
        cudaStream_t st = ctx->aux[jn++ % ctx->naux];
        long long blocks = (g.nunits - ctx->shard_rank + ctx->shard_n - 1) / ctx->shard_n;       // units owned by this rank
        if (blocks <= 0) continue;
        blocks = std::min<long long>(blocks, (long long)ctx->sm_count * g.ctas_per_sm);
        cudaError_t e = cudaSuccess;
        bool semi = false;                              // a job of the group stores or replays: the kernel variant with those paths
        for (const Shell4Job& hj : g.host_jobs) semi |= hj.store_mode != S4_DIRECT;
#define TUNA_MULTI4(GV) e = semi ? launch_shell4_multi<GV, true>(ctx, g, D, nD, Pc, Psym, Jc, Kc, tau, st, blocks) \
                                 : launch_shell4_multi<GV, false>(ctx, g, D, nD, Pc, Psym, Jc, Kc, tau, st, blocks);
        switch (g.G) {
            case 1: TUNA_MULTI4(1) break;
            case 2: TUNA_MULTI4(2) break;
            case 4: TUNA_MULTI4(4) break;
            case 8: TUNA_MULTI4(8) break;
            case 16: TUNA_MULTI4(16) break;
            case 32: TUNA_MULTI4(32) break;
            case 64: TUNA_MULTI4(64) break;
            case 128: TUNA_MULTI4(128) break;
            default: TUNA_MULTI4(256) break;
        }
#undef TUNA_MULTI4
        ctx->launches++;
        if (e != cudaSuccess) FAIL(TUNA_ERR_CUDA, std::string("k_shell4_multi launch: ") + cudaGetErrorString(e));
    }
    for (int a = 0; a < ctx->naux; ++a) {
        CK(cudaEventRecord(ctx->ev_join[a], ctx->aux[a]));
        CK(cudaStreamWaitEvent(ctx->stream, ctx->ev_join[a], 0));
    }
    // the store pass is enqueued: later builds (stream-ordered behind it) replay those jobs
    for (size_t j = 0; j < JS.jobs.size(); ++j) {
        if (modes[j] == S4_REPLAY) ctx->store_served = true;
        if (modes[j] != S4_STORE) continue;
        for (auto& e : ctx->store)
            if (e.cb == JS.jobs[j].cb && e.ck == JS.jobs[j].ck) e.filled = true;
    }
    return TUNA_OK;
}

// Direct mode on DEVICE buffers, in two halves that tuna_jk_direct_group runs on different devices.
// jk_direct_accumulate: P_cart = U^T P U, then the shell engine's integer accumulators d_fix (the per-component kernel: d_Jc / d_Kc).
// jk_direct_finish: J = U (Jacc + Jacc^T) U^T, K = U (Kacc +- Kacc^T) U^T from those accumulators; bit d of anti_mask marks density d as
// antisymmetric (its K is Kacc - Kacc^T and its J vanishes); all others must be symmetric.
static int jk_direct_accumulate(tuna_ctx* ctx, int nD, const double* dP, double tau) {
    const int nc = ctx->ncart, nb = ctx->nbf;
    const bool shell = ctx->direct_engine == 1 && ctx->ss.ok;
    int rc;
    if ((rc = ensure_mats(ctx, nD, nb, nc))) return rc;
    if ((rc = ensure_schwarz(ctx))) return rc;
    if (shell && (rc = ensure_shell4(ctx, tau, nD))) return rc;
    const size_t ncc = (size_t)nc * nc;
    const CsrDev& Uin = shell ? ctx->Uft : ctx->Ut;      // the shell engine works with unnormalised components: U' = U diag(f)
    // P_cart = U^T P U
    if ((rc = rotate(ctx, Uin, dP, ctx->d_tmp, nD, nb))) return rc;                          // [d][a][q] = sum_p U[p,a] P[d][p][q]
    if ((rc = rotate(ctx, Uin, ctx->d_tmp, ctx->d_Pc, (int64_t)nD * nc, 1))) return rc;      // [d][a][b] = sum_q U[q,b] tmp[d][a][q]
    CK(cudaMemsetAsync(ctx->d_scalars, 0, 2 * sizeof(unsigned long long), ctx->stream));
    if (shell) {
        CK(cudaMemsetAsync(ctx->d_eval, 0, sizeof(double), ctx->stream));
        k_absmax_scaled<<<grid_for(ctx, (int64_t)nD * ncc, 256, 4), 256, 0, ctx->stream>>>(ctx->d_Pc, ctx->d_finv, nc, nD, ctx->d_scalars);
    } else {
        k_absmax<<<grid_for(ctx, (int64_t)nD * ncc, 256, 4), 256, 0, ctx->stream>>>(ctx->d_Pc, (int64_t)nD * ncc, ctx->d_scalars);
    }
    ctx->launches++;
    const bool fixed = shell;        // the shell engine accumulates order-independently in integers; the per-component kernel uses FP64 atomics
    const size_t nacc = (size_t)nD * ncc;
    if (fixed) {
        GROW(ctx->d_fix, 4 * nacc);
        CK(cudaMemsetAsync(ctx->d_fix, 0, 4 * nacc * sizeof(long long), ctx->stream));
    } else {
        CK(cudaMemsetAsync(ctx->d_Jc, 0, nacc * sizeof(double), ctx->stream));
        CK(cudaMemsetAsync(ctx->d_Kc, 0, nacc * sizeof(double), ctx->stream));
    }
    CK(cudaEventRecord(ctx->ev[3][0], ctx->stream));
    if (shell) {
        k_add_transpose_signed<<<grid_for(ctx, (int64_t)nD * ncc, 256, 8), 256, 0, ctx->stream>>>(ctx->d_Pc, ctx->d_tmp, nD, nc, 0u);   // Psym = P + P^T
        ctx->launches++;
        double* Jw = reinterpret_cast<double*>(ctx->d_fix.get());
        double* Kw = reinterpret_cast<double*>(ctx->d_fix + 2 * nacc);
        if ((rc = launch_shell4_jobs(ctx, nD, ctx->d_Pc, ctx->d_tmp, Jw, Kw, tau, (long long)nacc))) return rc;
    } else {
        k_jk_direct<<<grid_for(ctx, ctx->task_begin[4] / ctx->shard_n + 1, 128, 16), 128, 0, ctx->stream>>>(
            table_dev(ctx), ctx->d_boys, ctx->d_herm, ctx->d_Q, ctx->d_Pc, ctx->d_Jc, ctx->d_Kc, nc, nD, tau, ctx->d_scalars, ctx->d_scalars + 1,
            ctx->shard_rank, ctx->shard_n);
        ctx->launches++;
        CK(cudaGetLastError());
    }
    CK(cudaEventRecord(ctx->ev[3][1], ctx->stream));
    return TUNA_OK;
}

static int jk_direct_finish(tuna_ctx* ctx, int nD, unsigned anti_mask, double* dJ, double* dK) {
    const int nc = ctx->ncart, nb = ctx->nbf;
    const bool shell = ctx->direct_engine == 1 && ctx->ss.ok;
    const size_t ncc = (size_t)nc * nc, nacc = (size_t)nD * ncc;
    const CsrDev& Uout = shell ? ctx->Uf : ctx->U;
    int rc;
    if (shell) {
        k_fixed_to_double<<<grid_for(ctx, (int64_t)nacc, 256, 8), 256, 0, ctx->stream>>>(ctx->d_fix, ctx->d_Jc, ctx->d_Kc, nacc);
        ctx->launches++;
    }
    for (int which = 0; which < 2; ++which) {
        double* acc = which == 0 ? ctx->d_Jc : ctx->d_Kc;
        double* out = which == 0 ? dJ : dK;
        if (!out) continue;
        k_add_transpose_signed<<<grid_for(ctx, (int64_t)nD * ncc, 256, 8), 256, 0, ctx->stream>>>(acc, ctx->d_Pc, nD, nc, which == 0 ? 0u : anti_mask);   // d_Pc reused as scratch
        ctx->launches++;
        if ((rc = rotate(ctx, Uout, ctx->d_Pc, ctx->d_tmp, nD, nc))) return rc;          // [d][p][b]
        if ((rc = rotate(ctx, Uout, ctx->d_tmp, out, (int64_t)nD * nb, 1))) return rc;    // [d][p][q]
    }
    CK(cudaGetLastError());
    return TUNA_OK;
}

// Densities are processed in passes small enough for the largest class of the basis to fit its J/K blocks in shared memory.
static int direct_pass_densities(const tuna_ctx* ctx, int nD) {
    int nd_max = 4;
    if (ctx->direct_engine == 1 && ctx->ss.ok) {
        int Lmax = 0;
        for (const auto& sh : ctx->ss.shells) Lmax = std::max(Lmax, sh.L);
        // staged densities + accumulators of the largest class: about 4 (nc + 4)^2 + 8 nc^2 doubles per density next to ~9000 doubles of tables
        const int nc = ctx->stab.nc[Lmax], per_density = 4 * (nc + 4) * (nc + 4) + 8 * nc * nc;
        while (nd_max > 1 && nd_max * per_density + 9000 > SHELL4_SMEM_DOUBLES) --nd_max;
    }
    const int npass = (nD + nd_max - 1) / nd_max;
    return (nD + npass - 1) / npass;
}

static int jk_direct_core(tuna_ctx* ctx, int nD, const double* dP, unsigned anti_mask, double* dJ, double* dK, double tau) {
    if (ctx->ncart == 0) FAIL(TUNA_ERR_STATE, "tuna_jk_direct: call tuna_set_basis first");
    if (ctx->nbf == 0) FAIL(TUNA_ERR_STATE, "tuna_jk_direct: call tuna_set_transform first");
    if (nD <= 0 || nD > 16 || !dP) FAIL(TUNA_ERR_ARG, "tuna_jk_direct: bad arguments (1 <= nD <= 16)");
    const int per = direct_pass_densities(ctx, nD);
    const size_t nn = (size_t)ctx->nbf * ctx->nbf;
    ctx->store_served = false;
    for (int d0 = 0; d0 < nD; d0 += per) {
        const int nd = std::min(per, nD - d0);
        int rc = jk_direct_accumulate(ctx, nd, dP + d0 * nn, tau);
        if (!rc) rc = jk_direct_finish(ctx, nd, (anti_mask >> d0) & ((1u << nd) - 1u), dJ ? dJ + d0 * nn : nullptr, dK ? dK + d0 * nn : nullptr);
        if (rc) return rc;
    }
    if (ctx->store_served) ++ctx->store_replays;
    return TUNA_OK;
}

// Host densities -> ctx's pinned staging buffer h_pin, split as plan_density (density_split.hpp) decides.  Sets ctx->dens_bound.
static int stage_host_density(tuna_ctx* ctx, int nD, const double* P, int* nDrun, unsigned* anti_mask) {
    const int nb = ctx->nbf;
    const size_t nn = (size_t)nb * nb;
    double pmax, amax;
    density_extrema(P, nD, nb, &pmax, &amax);
    const DensityPlan plan = plan_density(nD, pmax, amax);
    ctx->dens_bound = plan.dens_bound;
    *nDrun = plan.nDrun;
    *anti_mask = plan.anti_mask;
    int rc;
    if ((rc = ensure_mats(ctx, *nDrun, nb, ctx->ncart))) return rc;
    double* hP = ctx->h_pin;
    if (*nDrun == nD) {
        std::memcpy(hP, P, (size_t)nD * nn * sizeof(double));
    } else {
        for (int d = 0; d < nD; ++d)
            for (int i = 0; i < nb; ++i)
                for (int j = 0; j < nb; ++j) {
                    const double x = P[d * nn + (size_t)i * nb + j], y = P[d * nn + (size_t)j * nb + i];
                    hP[d * nn + (size_t)i * nb + j] = 0.5 * (x + y);
                    hP[(nD + d) * nn + (size_t)i * nb + j] = 0.5 * (x - y);
                }
    }
    return TUNA_OK;
}

// Device densities (caller's dP, ctx's device and stream) -> ctx->d_P, planned exactly as stage_host_density: k_density_scan, one 16-byte
// read-back and stream synchronise for plan_density, then the split (k_density_split) or a copy.  Sets ctx->dens_bound.
static int stage_device_density(tuna_ctx* ctx, int nD, const double* dP, int* nDrun, unsigned* anti_mask) {
    const int nb = ctx->nbf;
    const size_t nn = (size_t)nb * nb;
    GROW(ctx->h_scan, (size_t)2);
    CK(cudaMemsetAsync(ctx->d_scalars + 2, 0, 2 * sizeof(unsigned long long), ctx->stream));
    k_density_scan<<<grid_for(ctx, (int64_t)nD * nn, 256, 4), 256, 0, ctx->stream>>>(dP, nD, nb, ctx->d_scalars + 2);
    ctx->launches++;
    CK(cudaGetLastError());
    CK(cudaMemcpyAsync(ctx->h_scan, ctx->d_scalars + 2, 2 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    double pmax, amax;
    std::memcpy(&pmax, ctx->h_scan.get(), sizeof(double));
    std::memcpy(&amax, ctx->h_scan.get() + 1, sizeof(double));
    const DensityPlan plan = plan_density(nD, pmax, amax);
    ctx->dens_bound = plan.dens_bound;
    *nDrun = plan.nDrun;
    *anti_mask = plan.anti_mask;
    int rc;
    if ((rc = ensure_mats(ctx, *nDrun, nb, ctx->ncart))) return rc;
    if (*nDrun == nD) {
        CK(cudaMemcpyAsync(ctx->d_P, dP, (size_t)nD * nn * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    } else {
        k_density_split<<<grid_for(ctx, (int64_t)nD * nn, 256, 8), 256, 0, ctx->stream>>>(dP, ctx->d_P, nD, nb);
        ctx->launches++;
        CK(cudaGetLastError());
    }
    return TUNA_OK;
}

// ctx->d_J / d_K of a split stack (2 nD densities, as staged by stage_device_density) -> the caller's device J = J[S] and K = K[S] + K[A].
static int unstage_device_results(tuna_ctx* ctx, int nD, double* dJ, double* dK) {
    const size_t count = (size_t)nD * ctx->nbf * ctx->nbf;
    if (dJ) CK(cudaMemcpyAsync(dJ, ctx->d_J, count * sizeof(double), cudaMemcpyDeviceToDevice, ctx->stream));
    if (dK) {
        k_add_into<<<grid_for(ctx, (int64_t)count, 256, 8), 256, 0, ctx->stream>>>(dK, ctx->d_K, ctx->d_K + count, count);
        ctx->launches++;
        CK(cudaGetLastError());
    }
    return TUNA_OK;
}

// ctx->d_J / d_K (nDrun densities, as staged by stage_host_density) -> the caller's J and K; adds K[A] to K[S] for a general P.
static int unstage_host_results(tuna_ctx* ctx, int nD, int nDrun, double* J, double* K) {
    const size_t nn = (size_t)ctx->nbf * ctx->nbf, bytes = (size_t)nDrun * nn * sizeof(double);
    double* hJ = ctx->h_pin + (size_t)nDrun * nn;
    double* hK = hJ + (size_t)nDrun * nn;
    if (J) CK(cudaMemcpyAsync(hJ, ctx->d_J, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    if (K) CK(cudaMemcpyAsync(hK, ctx->d_K, bytes, cudaMemcpyDeviceToHost, ctx->stream));
    CK(cudaStreamSynchronize(ctx->stream));
    if (J) std::memcpy(J, hJ, (size_t)nD * nn * sizeof(double));
    if (K) {
        std::memcpy(K, hK, (size_t)nD * nn * sizeof(double));
        if (nDrun > nD)
            for (size_t x = 0; x < (size_t)nD * nn; ++x) K[x] += hK[(size_t)nD * nn + x];
    }
    return TUNA_OK;
}

// ------------------------------------------------------------------------------------------------
// one direct build over several devices (tuna_jk_direct_group)
// ------------------------------------------------------------------------------------------------
// acc[i] += stage[i] + stage[stride + i] + ... (npeer terms, in rank order).  For the shell engine's integer words T is unsigned: the sum
// wraps exactly like the atomicAdd on unsigned long long of DevPolicy::accumulate, so N partial accumulators add up to the 1-device words.
template <typename T>
__global__ void k_fix_reduce(T* __restrict__ acc, const T* __restrict__ stage, size_t count, size_t stride, int npeer) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += (size_t)gridDim.x * blockDim.x) {
        T s = acc[i];
        for (int p = 0; p < npeer; ++p) s += stage[(size_t)p * stride + i];
        acc[i] = s;
    }
}

static int group_check(tuna_ctx* const* ctxs, int nctx) {
    if (!ctxs || nctx < 1 || !ctxs[0]) return TUNA_ERR_ARG;
    tuna_ctx* ctx = ctxs[0];
    if (nctx > 64) FAIL(TUNA_ERR_ARG, "tuna_jk_direct_group: at most 64 contexts");
    for (int r = 1; r < nctx; ++r) {
        if (!ctxs[r]) FAIL(TUNA_ERR_ARG, "tuna_jk_direct_group: context of rank " + std::to_string(r) + " is null");
        for (int q = 0; q < r; ++q) {
            if (ctxs[q] == ctxs[r]) FAIL(TUNA_ERR_ARG, "tuna_jk_direct_group: ranks " + std::to_string(q) + " and " + std::to_string(r) + " are the same context");
            if (ctxs[q]->device == ctxs[r]->device)
                FAIL(TUNA_ERR_ARG, "tuna_jk_direct_group: ranks " + std::to_string(q) + " and " + std::to_string(r) + " are both on device " + std::to_string(ctxs[r]->device));
        }
    }
    if (ctx->ncart == 0 || ctx->nbf == 0) FAIL(TUNA_ERR_STATE, "tuna_jk_direct_group: basis and transform must be set first");
    for (int r = 0; r < nctx; ++r) {
        const tuna_ctx* c = ctxs[r];
        if (c->ncart != ctx->ncart || c->nbf != ctx->nbf || c->basis_sum != ctx->basis_sum || c->U_sum != ctx->U_sum || c->direct_engine != ctx->direct_engine)
            FAIL(TUNA_ERR_STATE, "tuna_jk_direct_group: rank " + std::to_string(r) + " holds a different basis or transform than rank 0");
        if (c->shard_rank != r || c->shard_n != nctx)
            FAIL(TUNA_ERR_STATE, "tuna_jk_direct_group: rank " + std::to_string(r) + " is sharded as (" + std::to_string(c->shard_rank) + ", " +
                                 std::to_string(c->shard_n) + "), expected (" + std::to_string(r) + ", " + std::to_string(nctx) + ")");
    }
    return TUNA_OK;
}

// One rank's accumulate half, enqueued from its own host thread; a peer then records ev_group for ctxs[0] to wait on.
static int group_accumulate(tuna_ctx* ctx, int nD, const double* dP, double tau, bool peer) try {
    CK(cudaSetDevice(ctx->device));
    if (int rc = jk_direct_accumulate(ctx, nD, dP, tau)) return rc;
    if (peer) CK(cudaEventRecord(ctx->ev_group, ctx->stream));
    return TUNA_OK;
} TUNA_CATCH

// dP, dJ, dK on ctxs[0]'s device; group_check has passed and every rank's dens_bound is set.
static int jk_direct_group_core(tuna_ctx* const* ctxs, int nctx, int nD, const double* dP, unsigned anti_mask, double* dJ, double* dK, double tau) {
    tuna_ctx* ctx = ctxs[0];
    if (nctx == 1) return jk_direct_core(ctx, nD, dP, anti_mask, dJ, dK, tau);
    if (nD <= 0 || nD > 16 || !dP) FAIL(TUNA_ERR_ARG, "tuna_jk_direct_group: bad arguments (1 <= nD <= 16)");
    const int nc = ctx->ncart, nb = ctx->nbf, npeer = nctx - 1;
    const bool fixed = ctx->direct_engine == 1 && ctx->ss.ok;
    const int per = direct_pass_densities(ctx, nD);
    const size_t nn = (size_t)nb * nb;
    int rc;
    for (int r = 0; r < nctx; ++r) ctxs[r]->store_served = false;
    for (int d0 = 0; d0 < nD; d0 += per) {
        const int nd = std::min(per, nD - d0);
        const size_t nacc = (size_t)nd * nc * nc, words = fixed ? 4 * nacc : 2 * nacc;     // one rank's accumulators
        const double* P0 = dP + d0 * nn;
        // 1. the pass's densities to every peer, after whatever produced them on ctxs[0]'s stream
        CK(cudaEventRecord(ctx->ev_group, ctx->stream));
        for (int r = 1; r < nctx; ++r) {
            tuna_ctx* c = ctxs[r];
            const unsigned long long bit = 1ull << (c->device & 63);
            if (!(ctx->peers_tried & bit)) {      // direct peer copies where the link allows them; without, the copies go through the host
                int ab = 0, ba = 0;
                CK(cudaDeviceCanAccessPeer(&ab, ctx->device, c->device));
                CK(cudaDeviceCanAccessPeer(&ba, c->device, ctx->device));
                if (ab && ba) {
                    CK(cudaSetDevice(ctx->device));
                    cudaDeviceEnablePeerAccess(c->device, 0);      // "already enabled" (e.g. by torch) or a refusal only costs speed
                    cudaGetLastError();
                    CK(cudaSetDevice(c->device));
                    cudaDeviceEnablePeerAccess(ctx->device, 0);
                    cudaGetLastError();
                }
                ctx->peers_tried |= bit;
            }
            CK(cudaSetDevice(c->device));
            if ((rc = ensure_mats(c, nd, nb, nc))) { ctx->err = "rank " + std::to_string(r) + ": " + c->err; return rc; }
            CK(cudaStreamWaitEvent(c->stream, ctx->ev_group, 0));
            CK(cudaMemcpyPeerAsync(c->d_P, c->device, P0, ctx->device, (size_t)nd * nn * sizeof(double), c->stream));
        }
        // 2. accumulate on every rank, enqueued from one host thread per device (all joined here)
        std::vector<int> rcs(nctx, TUNA_OK);
        {
            std::vector<std::thread> threads;
            try {
                for (int r = 1; r < nctx; ++r)
                    threads.emplace_back([&rcs, ctxs, r, nd, tau] { rcs[r] = group_accumulate(ctxs[r], nd, ctxs[r]->d_P, tau, true); });
            } catch (const std::exception& e) {
                for (auto& t : threads) t.join();
                FAIL(TUNA_ERR_STATE, std::string("tuna_jk_direct_group: cannot start a host thread: ") + e.what());
            }
            rcs[0] = group_accumulate(ctx, nd, P0, tau, false);
            for (auto& t : threads) t.join();
        }
        for (int r = 0; r < nctx; ++r)
            if (rcs[r]) {
                if (r > 0) ctx->err = "rank " + std::to_string(r) + ": " + ctxs[r]->err;
                return rcs[r];
            }
        CK(cudaSetDevice(ctx->device));
        // 3. pull every peer's accumulators into the staging buffer once its accumulate is done (one auxiliary stream per peer)
        if (ctx->d_peer.capacity() < npeer * words) {
            CK(cudaStreamSynchronize(ctx->stream));
            GROW(ctx->d_peer, npeer * words);
        }
        for (int r = 1; r < nctx; ++r) CK(cudaStreamWaitEvent(ctx->stream, ctxs[r]->ev_group, 0));
        CK(cudaEventRecord(ctx->ev[6][0], ctx->stream));
        for (int r = 1; r < nctx; ++r) {
            const tuna_ctx* c = ctxs[r];
            cudaStream_t st = ctx->aux[(r - 1) % tuna_ctx::NAUX];
            cudaEvent_t done = ctx->ev_join[(r - 1) % tuna_ctx::NAUX];
            long long* dst = ctx->d_peer + (size_t)(r - 1) * words;
            CK(cudaStreamWaitEvent(st, ctx->ev[6][0], 0));
            if (fixed) {
                CK(cudaMemcpyPeerAsync(dst, ctx->device, c->d_fix, c->device, words * sizeof(long long), st));
            } else {
                CK(cudaMemcpyPeerAsync(dst, ctx->device, c->d_Jc, c->device, nacc * sizeof(double), st));
                CK(cudaMemcpyPeerAsync(dst + nacc, ctx->device, c->d_Kc, c->device, nacc * sizeof(double), st));
            }
            CK(cudaEventRecord(done, st));
            CK(cudaStreamWaitEvent(ctx->stream, done, 0));
        }
        // 6. (enqueued now) no peer overwrites its accumulators in a later pass or call before they are pulled
        CK(cudaEventRecord(ctx->ev_group, ctx->stream));
        for (int r = 1; r < nctx; ++r) {
            CK(cudaSetDevice(ctxs[r]->device));
            CK(cudaStreamWaitEvent(ctxs[r]->stream, ctx->ev_group, 0));
        }
        CK(cudaSetDevice(ctx->device));
        // 4. sum into ctxs[0]'s accumulators, 5. finish there
        if (fixed) {
            k_fix_reduce<<<grid_for(ctx, (int64_t)words, 256, 8), 256, 0, ctx->stream>>>(reinterpret_cast<unsigned long long*>(ctx->d_fix.get()),
                reinterpret_cast<const unsigned long long*>(ctx->d_peer.get()), words, words, npeer);
        } else {
            const double* stage = reinterpret_cast<const double*>(ctx->d_peer.get());
            k_fix_reduce<<<grid_for(ctx, (int64_t)nacc, 256, 8), 256, 0, ctx->stream>>>(ctx->d_Jc.get(), stage, nacc, words, npeer);
            k_fix_reduce<<<grid_for(ctx, (int64_t)nacc, 256, 8), 256, 0, ctx->stream>>>(ctx->d_Kc.get(), stage + nacc, nacc, words, npeer);
            ctx->launches++;
        }
        ctx->launches++;
        CK(cudaGetLastError());
        if ((rc = jk_direct_finish(ctx, nd, (anti_mask >> d0) & ((1u << nd) - 1u), dJ ? dJ + d0 * nn : nullptr, dK ? dK + d0 * nn : nullptr))) return rc;
        CK(cudaEventRecord(ctx->ev[6][1], ctx->stream));
    }
    for (int r = 0; r < nctx; ++r)
        if (ctxs[r]->store_served) ++ctxs[r]->store_replays;
    return TUNA_OK;
}

extern "C" {

int tuna_jk_direct_dev(tuna_ctx* ctx, int nD, const double* dP, double* dJ, double* dK, double tau) try {
    if (!ctx) return TUNA_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    return jk_direct_core(ctx, nD, dP, 0u, dJ, dK, tau);
} TUNA_CATCH

int tuna_jk_direct(tuna_ctx* ctx, int nD, const double* P, double* J, double* K, double tau) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (ctx->ncart == 0 || ctx->nbf == 0) FAIL(TUNA_ERR_STATE, "tuna_jk_direct: basis and transform must be set first");
    if (nD <= 0 || nD > 8 || !P) FAIL(TUNA_ERR_ARG, "tuna_jk_direct: bad arguments (1 <= nD <= 8)");
    CK(cudaSetDevice(ctx->device));
    int rc, nDrun;
    unsigned anti_mask;
    if ((rc = stage_host_density(ctx, nD, P, &nDrun, &anti_mask))) return rc;
    CK(cudaMemcpyAsync(ctx->d_P, ctx->h_pin, (size_t)nDrun * ctx->nbf * ctx->nbf * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    if ((rc = jk_direct_core(ctx, nDrun, ctx->d_P, anti_mask, J ? ctx->d_J.get() : nullptr, K ? ctx->d_K.get() : nullptr, tau))) return rc;
    return unstage_host_results(ctx, nD, nDrun, J, K);
} TUNA_CATCH

int tuna_jk_direct_group_dev(tuna_ctx* const* ctxs, int nctx, int nD, const double* dP, double* dJ, double* dK, double tau) {
    tuna_ctx* ctx = (ctxs && nctx >= 1) ? ctxs[0] : nullptr;
    try {
        if (int rc = group_check(ctxs, nctx)) return rc;
        CK(cudaSetDevice(ctx->device));
        for (int r = 1; r < nctx; ++r) ctxs[r]->dens_bound = ctx->dens_bound;
        return jk_direct_group_core(ctxs, nctx, nD, dP, 0u, dJ, dK, tau);
    } TUNA_CATCH
}

int tuna_jk_direct_group(tuna_ctx* const* ctxs, int nctx, int nD, const double* P, double* J, double* K, double tau) {
    tuna_ctx* ctx = (ctxs && nctx >= 1) ? ctxs[0] : nullptr;
    try {
        int rc, nDrun;
        if ((rc = group_check(ctxs, nctx))) return rc;
        if (nD <= 0 || nD > 8 || !P) FAIL(TUNA_ERR_ARG, "tuna_jk_direct_group: bad arguments (1 <= nD <= 8)");
        CK(cudaSetDevice(ctx->device));
        unsigned anti_mask;
        if ((rc = stage_host_density(ctx, nD, P, &nDrun, &anti_mask))) return rc;
        for (int r = 1; r < nctx; ++r) ctxs[r]->dens_bound = ctx->dens_bound;
        CK(cudaMemcpyAsync(ctx->d_P, ctx->h_pin, (size_t)nDrun * ctx->nbf * ctx->nbf * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
        if ((rc = jk_direct_group_core(ctxs, nctx, nDrun, ctx->d_P, anti_mask, J ? ctx->d_J.get() : nullptr, K ? ctx->d_K.get() : nullptr, tau))) return rc;
        return unstage_host_results(ctx, nD, nDrun, J, K);
    } TUNA_CATCH
}

int tuna_jk_direct_general_dev(tuna_ctx* ctx, int nD, const double* dP, double* dJ, double* dK, double tau) try {
    if (!ctx) return TUNA_ERR_ARG;
    if (ctx->ncart == 0 || ctx->nbf == 0) FAIL(TUNA_ERR_STATE, "tuna_jk_direct_general_dev: basis and transform must be set first");
    if (nD <= 0 || nD > 8 || !dP) FAIL(TUNA_ERR_ARG, "tuna_jk_direct_general_dev: bad arguments (1 <= nD <= 8)");
    CK(cudaSetDevice(ctx->device));
    int rc, nDrun;
    unsigned anti_mask;
    if ((rc = stage_device_density(ctx, nD, dP, &nDrun, &anti_mask))) return rc;
    if (nDrun == nD) return jk_direct_core(ctx, nD, ctx->d_P, anti_mask, dJ, dK, tau);
    if ((rc = jk_direct_core(ctx, nDrun, ctx->d_P, anti_mask, dJ ? ctx->d_J.get() : nullptr, dK ? ctx->d_K.get() : nullptr, tau))) return rc;
    return unstage_device_results(ctx, nD, dJ, dK);
} TUNA_CATCH

int tuna_jk_direct_group_general_dev(tuna_ctx* const* ctxs, int nctx, int nD, const double* dP, double* dJ, double* dK, double tau) {
    tuna_ctx* ctx = (ctxs && nctx >= 1) ? ctxs[0] : nullptr;
    try {
        int rc, nDrun;
        if ((rc = group_check(ctxs, nctx))) return rc;
        if (nD <= 0 || nD > 8 || !dP) FAIL(TUNA_ERR_ARG, "tuna_jk_direct_group_general_dev: bad arguments (1 <= nD <= 8)");
        CK(cudaSetDevice(ctx->device));
        unsigned anti_mask;
        if ((rc = stage_device_density(ctx, nD, dP, &nDrun, &anti_mask))) return rc;
        for (int r = 1; r < nctx; ++r) ctxs[r]->dens_bound = ctx->dens_bound;
        if (nDrun == nD) return jk_direct_group_core(ctxs, nctx, nD, ctx->d_P, anti_mask, dJ, dK, tau);
        if ((rc = jk_direct_group_core(ctxs, nctx, nDrun, ctx->d_P, anti_mask, dJ ? ctx->d_J.get() : nullptr, dK ? ctx->d_K.get() : nullptr, tau))) return rc;
        return unstage_device_results(ctx, nD, dJ, dK);
    } TUNA_CATCH
}

int tuna_get_counts(const tuna_ctx* c, int64_t counts[8]) {
    if (!c || !counts) return TUNA_ERR_ARG;
    tuna_ctx* ctx = const_cast<tuna_ctx*>(c);
    if (ctx->ncart > 0 && !ctx->pairs_ready) { cudaSetDevice(ctx->device); if (int rc = ensure_pairs(ctx)) return rc; }
    unsigned long long ev = 0;
    if (ctx->d_scalars) {
        cudaSetDevice(ctx->device);
        cudaStreamSynchronize(ctx->stream);
        cudaMemcpy(&ev, ctx->d_scalars + 1, sizeof(ev), cudaMemcpyDeviceToHost);
        if (ctx->direct_engine == 1 && ctx->ss.ok && ctx->d_eval) {
            cudaMemcpy(&ev, ctx->d_eval, sizeof(ev), cudaMemcpyDeviceToHost);      // the engine counts evaluated quartets in a 64-bit integer
        }
    }
    counts[0] = ctx->pt.npair; counts[1] = ctx->n_unique; counts[2] = ctx->n_surviving; counts[3] = ctx->n_primq;
    counts[4] = (int64_t)ev; counts[5] = ctx->launches; counts[6] = ctx->ncart; counts[7] = ctx->nbf;
    return TUNA_OK;
}

int tuna_last_kernel_ms(tuna_ctx* ctx, int which, float* ms) {
    if (!ctx || !ms || which < 0 || which > 6) return TUNA_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    CK(cudaStreamSynchronize(ctx->stream));
    CK(cudaEventElapsedTime(ms, ctx->ev[which][0], ctx->ev[which][1]));
    return TUNA_OK;
}

int tuna_algorithmic_flops(const tuna_ctx* c, double* eri_flops, double* digest) {
    if (!c) return TUNA_ERR_ARG;
    tuna_ctx* ctx = const_cast<tuna_ctx*>(c);
    if (ctx->ncart > 0 && !ctx->pairs_ready) { cudaSetDevice(ctx->device); if (int rc = ensure_pairs(ctx)) return rc; }
    if (eri_flops) *eri_flops = ctx->alg_eri_flops;
    if (digest) *digest = ctx->alg_digest_flops;
    return TUNA_OK;
}

int tuna_fp64_peak_probe(tuna_ctx* ctx, double* tflops) {
    if (!ctx || !tflops) return TUNA_ERR_ARG;
    CK(cudaSetDevice(ctx->device));
    DevBuf<double> d;
    GROW(d, (size_t)1);
    const int blocks = ctx->sm_count * 8, threads = 256, iters = 1 << 14;
    cudaEvent_t e0, e1;
    CK(cudaEventCreate(&e0)); CK(cudaEventCreate(&e1));
    // SUSTAINED rate: two warm-up launches, then back-to-back launches timed as one interval of >= 0.5 s (a 2 ms burst overstates what
    // a second-long Fock build can reach under the power cap)
    for (int rep = 0; rep < 2; ++rep) k_dfma_probe<<<blocks, threads, 0, ctx->stream>>>(d, iters, 0.999999);
    CK(cudaStreamSynchronize(ctx->stream));
    double best = 0.0;
    int nl = 64;
    for (int round = 0; round < 4; ++round) {
        CK(cudaEventRecord(e0, ctx->stream));
        for (int rep = 0; rep < nl; ++rep) k_dfma_probe<<<blocks, threads, 0, ctx->stream>>>(d, iters, 0.999999);
        CK(cudaEventRecord(e1, ctx->stream));
        CK(cudaStreamSynchronize(ctx->stream));
        float ms = 0;
        CK(cudaEventElapsedTime(&ms, e0, e1));
        ctx->launches += nl;
        best = (double)nl * blocks * threads * iters * 8 * 2 / (ms * 1e-3) * 1e-12;
        if (ms >= 500.0f) break;
        nl = (int)std::min(4096.0, std::ceil(nl * 600.0 / std::max(ms, 1.0f)));
    }
    cudaEventDestroy(e0); cudaEventDestroy(e1);
    *tflops = best;
    return TUNA_OK;
}

}  // extern "C"
