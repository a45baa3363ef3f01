/*
 * CPU ORACLE of the spin-unrestricted nuclear gradient of the J/K energy — test infrastructure only
 * (tests/test_grad_uhf_cpu.py, tests/test_grad_uhf_gpu.py; loaded through tests/grad_oracle_uhf.py).
 *
 * It includes the closed-shell gradient oracle tests/grad_oracle.c unchanged (and through it the pinned
 * oracle/jk_oracle.c) and reuses its Rys roots, shell records, tile lists, l <= 5 ERI twin and centre_grad().
 * oracle_jk_grad_uhf() below is the canonical quartet loop of oracle_jk_grad() with the spin-resolved weight
 * and the two pooled densities of the unrestricted screen.
 */
#include "grad_oracle.c"

/* Screen of the unrestricted gradient: dj pools |Dt| (the J term), ds pools max_s |Ds| (the K terms). */
static inline int screen_grad_uhf_ok(int nbas, const float *q, const float *dj, const float *ds, int i, int j, int k,
                                     int l, int do_j, int do_k, float cutoff)
{
    const float q_ijkl = q[(size_t)i * nbas + j] + q[(size_t)k * nbas + l];
    float d_large = -73.6f;
    if (do_j) d_large = fmaxf(d_large, dj[(size_t)i * nbas + j] + dj[(size_t)k * nbas + l]);
    if (do_k) {
        d_large = fmaxf(d_large, ds[(size_t)i * nbas + k] + ds[(size_t)j * nbas + l]);
        d_large = fmaxf(d_large, ds[(size_t)i * nbas + l] + ds[(size_t)j * nbas + k]);
    }
    return q_ijkl + d_large > cutoff;
}

/* Nuclear gradient of
 *     E_U = (j_factor/2) tr(Dt J[Dt]) - (k_factor/2) [tr(Da K[Da]) + tr(Db K[Db])]
 * for the kernel-side spin densities dm = [Da, Db] (2 x nao x nao, symmetric) and dt = Da + Db, accumulated
 * per shell into gshell (nbas x 3, zeroed by the caller).  Canonical quartets as oracle_jk_grad(); tile lists
 * on 2 log_max_dm (the larger of the maxima of log_dj and log_ds); quartet screen screen_grad_uhf_ok(); weight
 * per component W_n = s (4 j_factor Dt_ij Dt_kl - 2 k_factor sum_s (Ds_ik Ds_jl + Ds_il Ds_jk)) with the
 * permutation factor s in the integral prefactor.  All four centres are evaluated.  Returns the number of
 * quartets evaluated. */
long oracle_jk_grad_uhf(int nbas, const double *rec, const int *angs, const int *nprims, const int *ao_loc,
                        const float *q, const float *log_dj, const float *log_ds, float log_max_dm, const double *dm,
                        const double *dt, double j_factor, double k_factor, double omega, float log_cutoff,
                        double *gshell)
{
    const int nao = ao_loc[nbas];
    const size_t nao2 = (size_t)nao * nao;
    const int do_j = j_factor != 0.0, do_k = k_factor != 0.0;
    uint8_t *tok = tile_mask(nbas, q, 2.0f * log_max_dm);
    const int nt = nbas / TILE;
    long total = 0;
    int nthreads = 1;
#ifdef _OPENMP
    nthreads = omp_get_max_threads();
#endif
    double *pg = (double *)calloc((size_t)nbas * 3 * nthreads, sizeof(double));
    const long npair = (long)nbas * (nbas + 1) / 2;
#pragma omp parallel reduction(+ : total)
    {
        int tid = 0;
#ifdef _OPENMP
        tid = omp_get_thread_num();
#endif
        double *mg = pg + (size_t)nbas * 3 * tid;
        const size_t nblk = (size_t)NFMAX5 * NFMAX5 * NFMAX5 * NFMAX5;
        double *W = (double *)malloc(sizeof(double) * nblk);
        double *blkp = (double *)malloc(sizeof(double) * nblk);
        double *blkm = (double *)malloc(sizeof(double) * nblk);
#pragma omp for schedule(dynamic, 4)
        for (long ij = npair - 1; ij >= 0; ij--) {
            int i = (int)((sqrt(8.0 * ij + 1.0) - 1.0) * 0.5);
            while ((long)i * (i + 1) / 2 > ij) i--;
            while ((long)(i + 1) * (i + 2) / 2 <= ij) i++;
            const int j = (int)(ij - (long)i * (i + 1) / 2);
            if (!tok[(size_t)(i / TILE) * nt + j / TILE]) continue;
            if (q[(size_t)i * nbas + j] + 0.f <= -99.f) continue;
            shell_t si, sj, sk, sl;
            load_shell(rec, i, &si); load_shell(rec, j, &sj);
            for (int k = 0; k <= i; k++) {
                load_shell(rec, k, &sk);
                for (int l = 0; l <= k; l++) {
                    if ((long)i * nbas + j < (long)k * nbas + l) continue;
                    if (!tok[(size_t)(k / TILE) * nt + l / TILE]) continue;
                    if (!screen_grad_uhf_ok(nbas, q, log_dj, log_ds, i, j, k, l, do_j, do_k, log_cutoff)) continue;
                    load_shell(rec, l, &sl);
                    double fac = PI_FAC;
                    if (i == j) fac *= .5;
                    if (k == l) fac *= .5;
                    if (i == k && j == l) fac *= .5;
                    const int ang[4] = {angs[i], angs[j], angs[k], angs[l]};
                    const int np[4] = {nprims[i], nprims[j], nprims[k], nprims[l]};
                    const int nfi = nf_of(ang[0]), nfj = nf_of(ang[1]), nfk = nf_of(ang[2]), nfl = nf_of(ang[3]);
#define DA_(r, c) dm[(size_t)(r) * nao + (c)]
#define DB_(r, c) dm[nao2 + (size_t)(r) * nao + (c)]
#define DT_(r, c) dt[(size_t)(r) * nao + (c)]
                    for (int a = 0; a < nfi; a++)
                    for (int b = 0; b < nfj; b++)
                    for (int c = 0; c < nfk; c++)
                    for (int e = 0; e < nfl; e++) {
                        const int ia = si.ao + a, jb = sj.ao + b, kc = sk.ao + c, le = sl.ao + e;
                        W[((a * nfj + b) * nfk + c) * nfl + e] =
                            4.0 * j_factor * DT_(ia, jb) * DT_(kc, le) -
                            2.0 * k_factor * ((DA_(ia, kc) * DA_(jb, le) + DA_(ia, le) * DA_(jb, kc)) +
                                              (DB_(ia, kc) * DB_(jb, le) + DB_(ia, le) * DB_(jb, kc)));
                    }
#undef DA_
#undef DB_
#undef DT_
                    const shell_t *sh[4] = {&si, &sj, &sk, &sl};
                    const int ids[4] = {i, j, k, l};
                    for (int c = 0; c < 4; c++) {
                        double g[3] = {0.0, 0.0, 0.0};
                        centre_grad(sh, ang, np, c, omega, fac, W, blkp, blkm, g);
                        for (int d = 0; d < 3; d++) mg[3 * ids[c] + d] += g[d];
                    }
                    total++;
                }
            }
        }
        free(W); free(blkp); free(blkm);
    }
    for (int t = 0; t < nthreads; t++)
        for (size_t n = 0; n < (size_t)nbas * 3; n++) gshell[n] += pg[(size_t)nbas * 3 * t + n];
    free(pg); free(tok);
    return total;
}
