/*
 * joltqc_b200 — C ABI of the B200-native FP64 direct-SCF J/K engine.
 *
 * This is the drop-in boundary for the one path this repository accelerates: the
 * Coulomb/exchange build behind jqc.pyscf.apply(mf) -> mf.get_jk(mol, dm, hermi, ...)
 * of ByteDance-Seed/JoltQC.  Every entry point names the reference interface it replaces
 * (paths relative to the reference repository).  Plain pointers and sizes only; device
 * pointers are CUDA device addresses on the engine's GPU.  All functions return 0 on
 * success or a negative JQC_E* code; jqc_last_error() gives the message (thread-local).
 * No exceptions cross this boundary and there is no CPU fallback: without a CUDA device
 * jqc_engine_create fails with JQC_ECUDA.
 */
#ifndef JOLTQC_B200_H
#define JOLTQC_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define JQC_OK 0
#define JQC_EINVAL (-1)   /* bad argument (shape, l > 4, nprim > 3, omega < 0, ...) */
#define JQC_ECUDA (-2)    /* CUDA runtime failure, no device */
#define JQC_ENOMEM (-3)
#define JQC_ESTATE (-4)   /* call order (e.g. finalize without a build) */

#define JQC_LMAX 4          /* jqc/constants.py:21 */
#define JQC_NPRIM_MAX 3     /* jqc/constants.py:24 */
#define JQC_BASIS_STRIDE 12 /* jqc/constants.py:27 */
#define JQC_TILE 4          /* jqc/constants.py:33 */

typedef struct jqc_engine jqc_engine;

/* Shell table in the reference's kernel-side layout (BasisLayout, jqc/pyscf/basis.py:66-480,
 * produced by split_basis :678-837 and sort_group_basis :483-675).  All arrays are HOST
 * pointers and are copied. */
typedef struct jqc_basis_desc {
    int nbas;                 /* padded shell count, multiple of JQC_TILE, <= 57344 (the reference allows 65535, jk.py:43-45) */
    const double* records;    /* nbas x 12: x,y,z,ao_loc,c0,e0,c1,e1,c2,e2,0,0 (basis.py:326-371) */
    const int* angs;          /* nbas */
    const int* nprims;        /* nbas */
    const int* ao_loc;        /* nbas + 1, kernel-side cartesian AO offsets; pads have zero width */
    const uint8_t* pad;       /* nbas, 1 for padding shells (basis.py:598-603) */
    int ngroups;              /* (l, nprim) groups, l ascending / nprim descending */
    const int* group_offset;  /* ngroups + 1 shell offsets, multiples of JQC_TILE */
    const int* mol_ao_offset; /* nbas: first molecular AO of the shell's parent, -1 for pads
                                 (BasisLayout.mol_ao_loc, basis.py:161-187) */
    int mol_nao;              /* AO count of the molecule (dm.shape[-1]) */
    int mol_cart;             /* 1: molecule uses cartesian AOs (cart2cart path), 0: real spherical */
    const double* c2s;        /* concatenated cart->sph matrices for l = 0..4, each row-major
                                 (ncart x (2l+1)); ignored when mol_cart (cart2sph.cu:22-100) */
} jqc_basis_desc;

/* Replaces BasisLayout.from_mol + generate_jk_kernel's captured state
 * (jqc/pyscf/__init__.py:188-226, jqc/pyscf/jk.py:93-107).  `device` is a CUDA ordinal. */
int jqc_engine_create(const jqc_basis_desc* desc, int device, jqc_engine** out);
void jqc_engine_destroy(jqc_engine* eng);
const char* jqc_last_error(void);

/* Static work partition for multi-GPU builds (SURVEY 8e; the reference is single-GPU,
 * README.md:104): this engine evaluates only the tasks assigned to `rank` of `world` -- a
 * deterministic interleave of the Schwarz-sorted task lists whose direction alternates from
 * round to round, so that every rank receives the same mix of heavy and light tasks.  The
 * caller sums the partial buffers of all ranks (one NCCL allreduce). */
int jqc_engine_set_shard(jqc_engine* eng, int rank, int world);

/* log-Schwarz matrix q[i,j] = log(sqrt(max|(ab|ab)|)+1e-300), float32 (nbas x nbas), pads
 * -100; evaluated on the GPU and cached per omega.  Replaces compute_q_matrix /
 * BasisLayout.q_matrix (jqc/pyscf/basis.py:218-243, 840-867; libcint on the CPU there).
 * *q_dev receives a device pointer owned by the engine. */
int jqc_q_matrix(jqc_engine* eng, double omega, const float** q_dev);

/* AO-basis transforms, device buffers.  Replace BasisLayout.dm_from_mol / dm_to_mol
 * (jqc/pyscf/basis.py:419-480; kernels jqc/backend/common/{sph2cart,cart2sph}.cu and the
 * Python cart2cart loop jqc/backend/cart2sph.py:241-307).
 * mol: (n, mol_nao, mol_nao), kernel side: (n, nao, nao), both C-order FP64. */
int jqc_dm_from_mol(jqc_engine* eng, const double* mol_dev, int n, double* kern_dev, void* stream);
int jqc_dm_to_mol(jqc_engine* eng, const double* kern_dev, int n, double* mol_dev, void* stream);

/* The operator: get_jk(mol, dm, hermi, vhfopt, with_j, with_k, omega, verbose)
 * (closure at jqc/pyscf/jk.py:109-382).  dm_dev: (n_dm, mol_nao, mol_nao) FP64 in the
 * molecule's AO basis.  vj_dev / vk_dev: same shape, written (not accumulated); pass NULL
 * for the one not requested (the reference returns the int 0 there).  hermi == 1 promises a
 * symmetric dm.  omega: 0 Coulomb, > 0 long-range erf (jk.py:133-134), < 0 -> JQC_EINVAL.
 * cutoff_fp64 / cutoff_fp32: the two screening thresholds of generate_jk_kernel
 * (jk.py:93-96; selection rule screen_jk_tasks.cu:258-261): quartets with estimate above
 * cutoff_fp32 are evaluated; those not above cutoff_fp64 form the FP32 band and are evaluated in
 * single precision with FP64 accumulation (jk.py:241-328) for the angular classes that have an FP32
 * kernel (every class up to f shells, and g-shell classes with blocks <= 108 elements; one density
 * matrix, hermi == 1), in FP64 otherwise.  With
 * cutoff_fp64 <= cutoff_fp32 (the default 1e-13 / 1e-13) the build is FP64 only.
 * Work is enqueued on `stream` (cudaStream_t, NULL = default stream); the call performs one host
 * synchronisation before the heavy kernels are enqueued (active tile counts), none afterwards;
 * results are complete when the stream reaches this point. */
int jqc_get_jk(jqc_engine* eng, const double* dm_dev, int n_dm, int hermi, int with_j, int with_k,
               double omega, double cutoff_fp64, double cutoff_fp32, double* vj_dev, double* vk_dev,
               void* stream);

/* Same operator with HOST buffers (pageable or pinned): copies dm in, runs, copies J/K out
 * and synchronises.  This is the end-to-end call bench.py times as `e2e`. */
int jqc_get_jk_host(jqc_engine* eng, const double* dm_host, int n_dm, int hermi, int with_j, int with_k,
                    double omega, double cutoff_fp64, double cutoff_fp32, double* vj_host, double* vk_host);

/* Two-phase form for multi-GPU: jqc_build_partial accumulates this rank's share into the
 * engine-owned kernel-side buffer [J || K] (2 * n_eff * nao * nao doubles, n_eff = n_dm or
 * 2 n_dm when hermi != 1; unused halves are zero) and returns its device pointer and length
 * for the caller's allreduce; jqc_finalize applies the reference's post-processing
 * (jk.py:353-370: scaling, transposes, back-transform) into vj_dev / vk_dev. */
int jqc_build_partial(jqc_engine* eng, const double* dm_dev, int n_dm, int hermi, int with_j, int with_k,
                      double omega, double cutoff_fp64, double cutoff_fp32, double** partial_dev,
                      size_t* partial_len, void* stream);
int jqc_finalize(jqc_engine* eng, double* vj_dev, double* vk_dev, void* stream);

/* Nuclear gradient of the J/K energy for one symmetric density D (molecule AO basis, FP64):
 *     E_jk(R) = (j_factor / 2) tr(D J[D]) - (k_factor / 4) tr(D K[D])
 * with J, K exactly what jqc_get_jk(hermi = 1, omega) returns; D is held fixed and the basis
 * functions move with their atoms.  grad_dev (natm x 3, device, Hartree/Bohr) is written with
 * g[A, x] = dE_jk / dR_{A,x}.  RHF: j_factor = k_factor = 1; hybrid: k_factor = hyb; the long-range
 * part of a range-separated hybrid is a second call with omega > 0, j_factor = 0,
 * k_factor = alpha - hyb.  shell_atom (HOST, nbas): atom of each kernel-side shell, -1 for pads.
 * Quartets are screened with q_ij + q_kl + max(d_ij + d_kl [j_factor != 0], d_ik + d_jl,
 * d_il + d_jk [k_factor != 0]) > log(cutoff) in float32 logs.  With a shard set
 * (jqc_engine_set_shard) the call writes this rank's partial gradient; the caller sums the ranks.
 * quartets (may be NULL): if given, the call synchronises and stores the number of quartets
 * evaluated.  JQC_EINVAL for omega < 0, j_factor == k_factor == 0, cutoff <= 0, natm < 1 or a
 * shell_atom entry outside [-1, natm).  The state of the last J/K build is left alone, so
 * jqc_build_partial -> jqc_jk_energy_grad -> jqc_finalize still finalises that build; scratch is
 * shared with the J/K builds, so calls on one engine are issued in stream order. */
int jqc_jk_energy_grad(jqc_engine* eng, const double* dm_dev, double j_factor, double k_factor,
                       double omega, double cutoff, const int* shell_atom, int natm, double* grad_dev,
                       long long* quartets, void* stream);

/* Spin-unrestricted form of jqc_jk_energy_grad for two symmetric spin densities Da, Db (dm_dev:
 * 2 x mol_nao x mol_nao, Da then Db, molecule AO basis, FP64) and Dt = Da + Db:
 *     E_U(R) = (j_factor / 2) tr(Dt J[Dt]) - (k_factor / 2) [tr(Da K[Da]) + tr(Db K[Db])]
 * with J, K exactly what jqc_get_jk(n_dm = 2, hermi = 1, omega) returns for [Da, Db]
 * (J[Dt] = J[Da] + J[Db]).  With Da = Db = D / 2 this is the E_jk(D) of jqc_jk_energy_grad.  One pass
 * over the derivative integrals serves both spins.  UHF: j_factor = k_factor = 1; UKS hybrid:
 * k_factor = hyb; the long-range part of a range-separated hybrid is a second call with omega > 0,
 * j_factor = 0, k_factor = alpha - hyb.  Quartets are screened with q_ij + q_kl + max(dJ_ij + dJ_kl
 * [j_factor != 0], dS_ik + dS_jl, dS_il + dS_jk [k_factor != 0]) > log(cutoff) in float32 logs, where
 * dJ pools |Dt| and dS pools max_s |Ds|.  grad_dev, shell_atom, natm, quartets, shards, JQC_EINVAL
 * cases and the untouched state of the last J/K build are as for jqc_jk_energy_grad. */
int jqc_jk_energy_grad_uhf(jqc_engine* eng, const double* dm_dev, double j_factor, double k_factor,
                           double omega, double cutoff, const int* shell_atom, int natm, double* grad_dev,
                           long long* quartets, void* stream);

/* Accounting of the last build (synchronises the engine's device).  counts: 625 entries,
 * quartets evaluated per class key ((li*5+lj)*5+lk)*5+ll; prim_weighted: the same weighted by
 * npi*npj*npk*npl (for the algorithmic FLOP model of SURVEY 8d); launches: kernels enqueued. */
int jqc_last_stats(jqc_engine* eng, long long* counts, long long* prim_weighted, int* launches);

/* Mixed-precision accounting of the last build: quartets[0] / quartets[1] = shell quartets evaluated
 * by the FP64 / FP32 kernels; ms (may be NULL) = their device times when profiling was enabled. */
int jqc_last_band_stats(jqc_engine* eng, long long* quartets, float* ms);

/* Per-class device time of the last build in ms (625 entries), measured with CUDA events
 * when profiling was enabled before the build (adds synchronisation; off by default). */
int jqc_set_profiling(jqc_engine* eng, int enabled);
int jqc_last_class_ms(jqc_engine* eng, float* ms);

/* Sizes derived from the table. */
int jqc_engine_nao(const jqc_engine* eng);
int jqc_engine_mol_nao(const jqc_engine* eng);

/* Measures the sustained FP64 FMA rate of the device with a register-resident DFMA loop
 * (roofline denominator measured on the box).  Returns TFLOP/s in *tflops. */
int jqc_fp64_peak_probe(int device, double* tflops, double* sm_clock_mhz);

#ifdef __cplusplus
}
#endif
#endif /* JOLTQC_B200_H */
