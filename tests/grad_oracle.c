/*
 * CPU ORACLE of the nuclear gradient of the J/K energy — test infrastructure only
 * (tests/test_grad_cpu.py, tests/test_grad_gpu.py; loaded through tests/grad_oracle.py).
 *
 * It includes the pinned J/K oracle oracle/jk_oracle.c unchanged and reuses its Rys roots, shell
 * records, canonical quartet order and tile lists.  The derivative integrals of all four centres come
 * from the identity  d phi / dR_x = 2a phi(l+1_x) - l_x phi(l-1_x):  plain ERI blocks of raised shells
 * (coefficients 2a c) and lowered shells, no derivative recurrences, so the result is independent of
 * the GPU construction (jk_grad.cuh).  Raised shells reach l = 5, beyond the array bounds of the pinned
 * eri_block(); eri_block_l5() below is the same routine with bounds for l = 5, and
 * tests/test_grad_cpu.py checks it against the pinned one on every class up to l = 4.
 */
#include "jk_oracle.c"

#define L1_5 6                 /* l + 1 for l = 5 */
#define LL2_5 11               /* 2 l + 1 for l = 5 */
#define NFMAX5 21              /* cartesian components of l = 5 */

/* ------------------------------------------------------------------ ERI block, l <= 5 */
/* eri_block() of jk_oracle.c, line for line, with array bounds for l = 5 */
static void eri_block_l5(const shell_t *si, const shell_t *sj, const shell_t *sk, const shell_t *sl,
                      int li, int lj, int lk, int ll, int npi, int npj, int npk, int npl,
                      double omega, double fac, double *out)
{
    const int lij = li + lj, lkl = lk + ll;
    const int nroots = (lij + lkl) / 2 + 1;
    const int nfi = nf_of(li), nfj = nf_of(lj), nfk = nf_of(lk), nfl = nf_of(ll);
    int ix[NFMAX5], iy[NFMAX5], iz[NFMAX5], jx[NFMAX5], jy[NFMAX5], jz[NFMAX5];
    int kx[NFMAX5], ky[NFMAX5], kz[NFMAX5], lx[NFMAX5], ly[NFMAX5], lz[NFMAX5];
    cart_xyz(li, ix, iy, iz); cart_xyz(lj, jx, jy, jz);
    cart_xyz(lk, kx, ky, kz); cart_xyz(ll, lx, ly, lz);

    double rjri[3], rlrk[3];
    double rr_ij = 0, rr_kl = 0;
    for (int d = 0; d < 3; d++) {
        rjri[d] = sj->r[d] - si->r[d]; rr_ij += rjri[d] * rjri[d];
        rlrk[d] = sl->r[d] - sk->r[d]; rr_kl += rlrk[d] * rlrk[d];
    }
    /* t[d][i][k], then g[d][i][j][k][l] */
    static _Thread_local double t[3][LL2_5][LL2_5];
    static _Thread_local double h[3][LL2_5][L1_5][LL2_5];
    static _Thread_local double g[3][L1_5][L1_5][L1_5][L1_5];
    double rw[2 * 16];

    for (int kp = 0; kp < npk; kp++)
    for (int lp = 0; lp < npl; lp++) {
        const double ak = sk->e[kp], al = sl->e[lp];
        const double akl = ak + al, inv_akl = 1.0 / akl;
        const double al_akl = al * inv_akl;
        const double Kcd = exp(-ak * al_akl * rr_kl);
        const double ckcl = sk->c[kp] * sl->c[lp] * Kcd;
        for (int ip = 0; ip < npi; ip++)
        for (int jp = 0; jp < npj; jp++) {
            const double ai = si->e[ip], aj = sj->e[jp];
            const double aij = ai + aj, inv_aij = 1.0 / aij;
            const double aj_aij = aj * inv_aij;
            const double Kab = exp(-ai * aj_aij * rr_ij);
            const double cicj = fac * si->c[ip] * sj->c[jp] * Kab;
            double Rpq[3], rr = 0;
            for (int d = 0; d < 3; d++) {
                const double pij = rjri[d] * aj_aij + si->r[d];
                const double pkl = rlrk[d] * al_akl + sk->r[d];
                Rpq[d] = pij - pkl; rr += Rpq[d] * Rpq[d];
            }
            const double inv_aijkl = 1.0 / (aij + akl);
            const double theta = aij * akl * inv_aijkl;
            const double gy0 = cicj * inv_aij * inv_akl * sqrt(inv_aijkl);
            rys_roots(nroots, rr, rw, theta, omega);
            for (int ir = 0; ir < nroots; ir++) {
                const double rt = rw[2 * ir];
                const double rt_aa = rt * inv_aijkl;
                const double rt_aij = rt_aa * akl, rt_akl = rt_aa * aij;
                const double b10 = .5 * inv_aij * (1.0 - rt_aij);
                const double b01 = .5 * inv_akl * (1.0 - rt_akl);
                const double b00 = .5 * rt_aa;
                const double seed[3] = {ckcl, gy0, rw[2 * ir + 1]};
                for (int d = 0; d < 3; d++) {
                    const double c0 = rjri[d] * aj_aij - rt_aij * Rpq[d];
                    const double cp = rlrk[d] * al_akl + rt_akl * Rpq[d];
                    /* TRR (1q1t.cu:244-330) */
                    t[d][0][0] = seed[d];
                    for (int i = 0; i < lij; i++)
                        t[d][i + 1][0] = c0 * t[d][i][0] + (i > 0 ? i * b10 * t[d][i - 1][0] : 0.0);
                    for (int k = 0; k < lkl; k++)
                        for (int i = 0; i <= lij; i++) {
                            double v = cp * t[d][i][k];
                            if (k > 0) v += k * b01 * t[d][i][k - 1];
                            if (i > 0) v += i * b00 * t[d][i - 1][k];
                            t[d][i][k + 1] = v;
                        }
                    /* HRR on the bra (1q1t.cu:336-358): g(i,j+1) = g(i+1,j) - (Rj-Ri) g(i,j) */
                    for (int k = 0; k <= lkl; k++) {
                        for (int i = 0; i <= lij; i++) h[d][i][0][k] = t[d][i][k];
                        for (int j = 0; j < lj; j++)
                            for (int i = 0; i <= lij - j - 1; i++)
                                h[d][i][j + 1][k] = h[d][i + 1][j][k] - rjri[d] * h[d][i][j][k];
                    }
                    /* HRR on the ket (1q1t.cu:360-382) */
                    for (int i = 0; i <= li; i++)
                        for (int j = 0; j <= lj; j++) {
                            double w[LL2_5][L1_5];
                            for (int k = 0; k <= lkl; k++) w[k][0] = h[d][i][j][k];
                            for (int l = 0; l < ll; l++)
                                for (int k = 0; k <= lkl - l - 1; k++)
                                    w[k][l + 1] = w[k + 1][l] - rlrk[d] * w[k][l];
                            for (int k = 0; k <= lk; k++)
                                for (int l = 0; l <= ll; l++) g[d][i][j][k][l] = w[k][l];
                        }
                }
                /* product (1q1t.cu:384-405) */
                double *o = out;
                for (int i = 0; i < nfi; i++)
                for (int j = 0; j < nfj; j++)
                for (int k = 0; k < nfk; k++)
                for (int l = 0; l < nfl; l++)
                    *o++ += g[0][ix[i]][jx[j]][kx[k]][lx[l]] * g[1][iy[i]][jy[j]][ky[k]][ly[l]] *
                            g[2][iz[i]][jz[j]][kz[k]][lz[l]];
            }
        }
    }
}

/* (ij|kl) cartesian block of eri_block_l5() for sorted-table shells (no symmetry factor): the
 * counterpart of oracle_eri_block(), for the pin against the pinned routine */
void grad_oracle_eri_block(const double *rec, const int *angs, const int *nprims,
                           int ish, int jsh, int ksh, int lsh, double omega, double *out)
{
    shell_t si, sj, sk, sl;
    load_shell(rec, ish, &si); load_shell(rec, jsh, &sj);
    load_shell(rec, ksh, &sk); load_shell(rec, lsh, &sl);
    const int n = nf_of(angs[ish]) * nf_of(angs[jsh]) * nf_of(angs[ksh]) * nf_of(angs[lsh]);
    memset(out, 0, sizeof(double) * n);
    eri_block_l5(&si, &sj, &sk, &sl, angs[ish], angs[jsh], angs[ksh], angs[lsh],
                 nprims[ish], nprims[jsh], nprims[ksh], nprims[lsh], omega, PI_FAC, out);
}

/* ------------------------------------------------------------------ energy gradient */
/* Screen of the J/K energy gradient: the weights are products of two density blocks. */
static inline int screen_grad_ok(int nbas, const float *q, const float *d, int i, int j, int k, int l,
                                 int do_j, int do_k, float cutoff)
{
    const float q_ijkl = q[(size_t)i * nbas + j] + q[(size_t)k * nbas + l];
    float d_large = -73.6f;
    if (do_j) d_large = fmaxf(d_large, d[(size_t)i * nbas + j] + d[(size_t)k * nbas + l]);
    if (do_k) {
        d_large = fmaxf(d_large, d[(size_t)i * nbas + k] + d[(size_t)j * nbas + l]);
        d_large = fmaxf(d_large, d[(size_t)i * nbas + l] + d[(size_t)j * nbas + k]);
    }
    return q_ijkl + d_large > cutoff;
}

/* index of the cartesian component (x, y, l - x - y) in the order of cart_xyz() */
static inline int cart_index(int l, int x, int y) { return (l - x) * (l - x + 1) / 2 + (l - x - y); }

/* out[3] += d/dR_c sum_n W_n (ij|kl)_n for centre c of the quartet, from the identity
 * d phi / dR_x = 2a phi(l+1_x) - l_x phi(l-1_x): the raised shell carries the coefficients 2a c, the
 * lowered one the plain coefficients; both blocks come from eri_block(). */
static void centre_grad(const shell_t *const sh[4], const int ang[4], const int np[4], int c, double omega, double fac,
                        const double *W, double *blkp, double *blkm, double out[3])
{
    int lx[4][NFMAX5], ly[4][NFMAX5], lz[4][NFMAX5], nf[4];
    for (int s = 0; s < 4; s++) { cart_xyz(ang[s], lx[s], ly[s], lz[s]); nf[s] = nf_of(ang[s]); }
    shell_t up = *sh[c];
    for (int p = 0; p < 3; p++) up.c[p] = 2.0 * up.e[p] * sh[c]->c[p];
    const shell_t *s4[4] = {sh[0], sh[1], sh[2], sh[3]};
    int lu[4] = {ang[0], ang[1], ang[2], ang[3]}, nfu[4];
    s4[c] = &up;
    lu[c] = ang[c] + 1;
    for (int s = 0; s < 4; s++) nfu[s] = nf_of(lu[s]);
    memset(blkp, 0, sizeof(double) * nfu[0] * nfu[1] * nfu[2] * nfu[3]);
    eri_block_l5(s4[0], s4[1], s4[2], s4[3], lu[0], lu[1], lu[2], lu[3], np[0], np[1], np[2], np[3], omega, fac, blkp);
    int ld[4] = {ang[0], ang[1], ang[2], ang[3]}, nfd[4];
    const int lower = ang[c] > 0;
    if (lower) {
        ld[c] = ang[c] - 1;
        for (int s = 0; s < 4; s++) nfd[s] = nf_of(ld[s]);
        memset(blkm, 0, sizeof(double) * nfd[0] * nfd[1] * nfd[2] * nfd[3]);
        eri_block_l5(sh[0], sh[1], sh[2], sh[3], ld[0], ld[1], ld[2], ld[3], np[0], np[1], np[2], np[3], omega, fac, blkm);
    }
    int idx[4];
    for (idx[0] = 0; idx[0] < nf[0]; idx[0]++)
    for (idx[1] = 0; idx[1] < nf[1]; idx[1]++)
    for (idx[2] = 0; idx[2] < nf[2]; idx[2]++)
    for (idx[3] = 0; idx[3] < nf[3]; idx[3]++) {
        const double w = W[((idx[0] * nf[1] + idx[1]) * nf[2] + idx[2]) * nf[3] + idx[3]];
        const int e[3] = {lx[c][idx[c]], ly[c][idx[c]], lz[c][idx[c]]};
        for (int d = 0; d < 3; d++) {
            int r[4] = {idx[0], idx[1], idx[2], idx[3]};
            r[c] = cart_index(lu[c], e[0] + (d == 0), e[1] + (d == 1));
            out[d] += w * blkp[((r[0] * nfu[1] + r[1]) * nfu[2] + r[2]) * nfu[3] + r[3]];
            if (e[d] > 0) {
                r[c] = cart_index(ld[c], e[0] - (d == 0), e[1] - (d == 1));
                out[d] -= w * e[d] * blkm[((r[0] * nfd[1] + r[1]) * nfd[2] + r[2]) * nfd[3] + r[3]];
            }
        }
    }
}

/* Nuclear gradient of E_jk = (j_factor/2) tr(D J[D]) - (k_factor/4) tr(D K[D]) for one symmetric
 * kernel-side density dm (nao x nao), accumulated per shell into gshell (nbas x 3, zeroed by the
 * caller).  Canonical quartets as oracle_build_jk; tile lists on 2 log max|D|; quartet screen
 * screen_grad_ok(); weight per component W_n = s (4 j_factor D_ij D_kl - k_factor (D_ik D_jl + D_il D_jk))
 * with the permutation factor s in the integral prefactor.  All four centres are evaluated.
 * Returns the number of quartets evaluated. */
long oracle_jk_grad(int nbas, const double *rec, const int *angs, const int *nprims, const int *ao_loc,
                    const float *q, const float *log_dm_cond, float log_max_dm, const double *dm,
                    double j_factor, double k_factor, double omega, float log_cutoff, double *gshell)
{
    const int nao = ao_loc[nbas];
    const int do_j = j_factor != 0.0, do_k = k_factor != 0.0;
    uint8_t *tok = tile_mask(nbas, q, 2.0f * log_max_dm);   /* exact doubling: log(1e-13) - 2 log max|D| */
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
                    if (!screen_grad_ok(nbas, q, log_dm_cond, i, j, k, l, do_j, do_k, log_cutoff)) continue;
                    load_shell(rec, l, &sl);
                    double fac = PI_FAC;
                    if (i == j) fac *= .5;
                    if (k == l) fac *= .5;
                    if (i == k && j == l) fac *= .5;
                    const int ang[4] = {angs[i], angs[j], angs[k], angs[l]};
                    const int np[4] = {nprims[i], nprims[j], nprims[k], nprims[l]};
                    const int nfi = nf_of(ang[0]), nfj = nf_of(ang[1]), nfk = nf_of(ang[2]), nfl = nf_of(ang[3]);
#define D_(r, c) dm[(size_t)(r) * nao + (c)]
                    for (int a = 0; a < nfi; a++)
                    for (int b = 0; b < nfj; b++)
                    for (int c = 0; c < nfk; c++)
                    for (int e = 0; e < nfl; e++) {
                        const int ia = si.ao + a, jb = sj.ao + b, kc = sk.ao + c, le = sl.ao + e;
                        W[((a * nfj + b) * nfk + c) * nfl + e] =
                            4.0 * j_factor * D_(ia, jb) * D_(kc, le) - k_factor * (D_(ia, kc) * D_(jb, le) + D_(ia, le) * D_(jb, kc));
                    }
#undef D_
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
