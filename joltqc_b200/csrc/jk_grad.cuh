// Nuclear gradient of the J/K energy, one quartet per thread over a quartet list (FP64).
//
// For a symmetric kernel-side density D the energy
//     E_jk = (j_factor / 2) tr(D J[D]) - (k_factor / 4) tr(D K[D])
// is a sum over the canonical quartets of W_n (ij|kl)_n with, per cartesian component n = (i,j,k,l),
//     W_n = 4 j_factor D_ij D_kl - k_factor (D_ik D_jl + D_il D_jk)
// (the permutation factor s of jk_1q1t_body.inc rides in the integral prefactor, as for J/K).
// The derivative with respect to the centre A of shell i is
//     d(ij|kl)/dA_x = 2 a (i+1_x j|kl) - i_x (i-1_x j|kl)
// and likewise for j and k; the centre of l follows from translational invariance.
//
// The Rys g arrays are filled for the shape (LI+1, LJ, LK+1, LL): TRR to bra total LIJ+1 and ket total
// LKL+1, then the usual HRR.  The raised j components come from the bra HRR identity
// (i, j+1) = (i+1, j) - (Rj - Ri) (i, j), so no second raised block is needed.  The contraction
// streams: per primitive quartet and root only nine partial sums (three centres x xyz) are kept; the
// 2a factors are applied per primitive quartet, the lowered terms (no exponent) once per quartet.
// Each quartet adds its four centres' 3-vectors into a per-shell nbas x 3 accumulator.
//
// NSPIN = 2 is the spin-unrestricted energy for two symmetric spin densities Da, Db (Dt = Da + Db)
//     E_U = (j_factor / 2) tr(Dt J[Dt]) - (k_factor / 2) [tr(Da K[Da]) + tr(Db K[Db])]
// with the weight
//     W_n = 4 j_factor Dt_ij Dt_kl - 2 k_factor sum_s (Ds_ik Ds_jl + Ds_il Ds_jk);
// everything downstream of the weight is the same as for NSPIN = 1.
#pragma once
#include "jk_1q1t.cuh"

namespace jqc {

struct GradArgs {
    int nao;
    int npi, npj, npk, npl;
    const double* __restrict__ basis;     // nbas x 12 packed shell records
    const double* __restrict__ dm;        // nao x nao kernel-side cartesian density (symmetric); NSPIN = 2: Da
    double j_factor4;                     // 4 * j_factor
    double k_factor;                      // k_factor; NSPIN = 2: 2 * k_factor
    double omega;                         // 0: Coulomb, > 0: long-range erf
    const ushort4* __restrict__ quartets;
    const unsigned* __restrict__ ntasks;  // device counter written by the task generator
    double* __restrict__ gshell;          // nbas x 3, accumulated
    const double* __restrict__ dm_b;      // NSPIN = 2: Db (nao x nao, symmetric)
    const double* __restrict__ dm_t;      // NSPIN = 2: Dt = Da + Db
};

// W_n of one cartesian component (absolute AO indices)
template <int NSPIN>
__device__ __forceinline__ double grad_weight(const GradArgs& a, int i, int j, int k, int l)
{
    const size_t n = (size_t)a.nao;
    if constexpr (NSPIN == 1) {
        const double* __restrict__ dm = a.dm;
        return fma(a.j_factor4 * __ldg(dm + i * n + j), __ldg(dm + k * n + l),
                   -a.k_factor * fma(__ldg(dm + i * n + k), __ldg(dm + j * n + l), __ldg(dm + i * n + l) * __ldg(dm + j * n + k)));
    } else {
        const double* __restrict__ da = a.dm;
        const double* __restrict__ db = a.dm_b;
        const double* __restrict__ dt = a.dm_t;
        const double ka = fma(__ldg(da + i * n + k), __ldg(da + j * n + l), __ldg(da + i * n + l) * __ldg(da + j * n + k));
        const double kb = fma(__ldg(db + i * n + k), __ldg(db + j * n + l), __ldg(db + i * n + l) * __ldg(db + j * n + k));
        return fma(a.j_factor4 * __ldg(dt + i * n + j), __ldg(dt + k * n + l), -a.k_factor * (ka + kb));
    }
}

template <int LI, int LJ, int LK, int LL>
struct GradShape {
    using S = QuartetShape<LI, LJ, LK, LL>;
    using G = QuartetShape<LI + 1, LJ, LK + 1, LL>;   // g layout with i and k raised by one
    static constexpr int NROOTS = (S::LIJ + S::LKL + 1) / 2 + 1;
    // fully unrolled (density weights formed once per quartet, weights and g arrays in registers) for
    // small classes; otherwise rolled, with the g arrays in thread-local scratch and each weight formed
    // where it is used (a stored block would cost up to 405 KB of stack per thread for (gg|gg))
    static constexpr bool SMALL = 3 * G::GSIZE + S::N <= 128;
};

template <int LI, int LJ, int LK, int LL, bool SMALL, int NT, int NSPIN>
__global__ void __launch_bounds__(NT) jk_grad_kernel(const GradArgs a)
{
    using S = QuartetShape<LI, LJ, LK, LL>;
    using G = typename GradShape<LI, LJ, LK, LL>::G;
    constexpr int NFI = S::NFI, NFJ = S::NFJ, NFK = S::NFK, NFL = S::NFL, N = S::N;
    constexpr int NROOTS = GradShape<LI, LJ, LK, LL>::NROOTS;
    constexpr int GS = G::GSIZE, DJ = G::DJ, DK = G::DK, DL = G::DL;
    constexpr int U = SMALL ? 64 : 1;   // unroll count: 64 exceeds every trip count (full unrolling)

    const unsigned ntasks = *a.ntasks;
#pragma unroll 1
    for (unsigned wbase = blockIdx.x * NT + (threadIdx.x & ~31u); wbase < ntasks; wbase += gridDim.x * NT) {
        const unsigned task = wbase + (threadIdx.x & 31u);
        const bool live = task < ntasks;
        const ushort4 sq = a.quartets[live ? task : wbase];
        const int ish = sq.x, jsh = sq.y, ksh = sq.z, lsh = sq.w;
        const double* __restrict__ bi = a.basis + ish * BASIS_STRIDE;
        const double* __restrict__ bj = a.basis + jsh * BASIS_STRIDE;
        const double* __restrict__ bk = a.basis + ksh * BASIS_STRIDE;
        const double* __restrict__ bl = a.basis + lsh * BASIS_STRIDE;
        const double4 ri = *reinterpret_cast<const double4*>(bi);
        const double4 rj = *reinterpret_cast<const double4*>(bj);
        const double4 rk = *reinterpret_cast<const double4*>(bk);
        const double4 rl = *reinterpret_cast<const double4*>(bl);

        double fac = live ? PI_FAC : 0.0;
        if (ish == jsh) fac *= 0.5;
        if (ksh == lsh) fac *= 0.5;
        if (ish == ksh && jsh == lsh) fac *= 0.5;

        const int i0 = (int)ri.w, j0 = (int)rj.w, k0 = (int)rk.w, l0 = (int)rl.w;
        double w[SMALL ? N : 1];
        if constexpr (SMALL) {
#pragma unroll
            for (int i = 0; i < NFI; i++)
#pragma unroll
            for (int j = 0; j < NFJ; j++)
#pragma unroll
            for (int k = 0; k < NFK; k++)
#pragma unroll
            for (int l = 0; l < NFL; l++) w[((i * NFJ + j) * NFK + k) * NFL + l] = grad_weight<NSPIN>(a, i0 + i, j0 + j, k0 + k, l0 + l);
        }

        const double rjri[3] = {rj.x - ri.x, rj.y - ri.y, rj.z - ri.z};
        const double rlrk[3] = {rl.x - rk.x, rl.y - rk.y, rl.z - rk.z};
        const double rr_ij = rjri[0] * rjri[0] + rjri[1] * rjri[1] + rjri[2] * rjri[2];
        const double rr_kl = rlrk[0] * rlrk[0] + rlrk[1] * rlrk[1] + rlrk[2] * rlrk[2];

        // gradient of centres i, j, k: raised terms (times 2a per primitive) and lowered terms
        double gi[3] = {0.0, 0.0, 0.0}, gj[3] = {0.0, 0.0, 0.0}, gk[3] = {0.0, 0.0, 0.0};
        double mi[3] = {0.0, 0.0, 0.0}, mj[3] = {0.0, 0.0, 0.0}, mk[3] = {0.0, 0.0, 0.0};

#pragma unroll 1
        for (int kp = 0; kp < a.npk; kp++)
#pragma unroll 1
        for (int lp = 0; lp < a.npl; lp++) {
            const double2 cek = *reinterpret_cast<const double2*>(bk + 4 + 2 * kp);
            const double2 cel = *reinterpret_cast<const double2*>(bl + 4 + 2 * lp);
            const double akl = cek.y + cel.y;
            const double inv_akl = 1.0 / akl;
            const double al_akl = cel.y * inv_akl;
            const double ckcl = cek.x * cel.x * exp(-cek.y * al_akl * rr_kl);
            const double qx = fma(rlrk[0], al_akl, rk.x), qy = fma(rlrk[1], al_akl, rk.y), qz = fma(rlrk[2], al_akl, rk.z);
#pragma unroll 1
            for (int ip = 0; ip < a.npi; ip++)
#pragma unroll 1
            for (int jp = 0; jp < a.npj; jp++) {
                const double2 cei = *reinterpret_cast<const double2*>(bi + 4 + 2 * ip);
                const double2 cej = *reinterpret_cast<const double2*>(bj + 4 + 2 * jp);
                const double aij = cei.y + cej.y;
                const double inv_aij = 1.0 / aij;
                const double aj_aij = cej.y * inv_aij;
                const double cicj = fac * cei.x * cej.x * exp(-cei.y * aj_aij * rr_ij);
                const double Rpq[3] = {fma(rjri[0], aj_aij, ri.x) - qx, fma(rjri[1], aj_aij, ri.y) - qy,
                                       fma(rjri[2], aj_aij, ri.z) - qz};
                const double rr = Rpq[0] * Rpq[0] + Rpq[1] * Rpq[1] + Rpq[2] * Rpq[2];
                const double inv_aijkl = 1.0 / (aij + akl);
                const double theta = aij * akl * inv_aijkl;
                const double gy0 = cicj * inv_aij * inv_akl * sqrt(inv_aijkl);
                double rw[2 * NROOTS];
                double theta_fac = 1.0, sqrt_theta_fac = 1.0;
                if (a.omega > 0.0) {
                    const double o2 = a.omega * a.omega;
                    theta_fac = o2 / (o2 + theta);
                    sqrt_theta_fac = sqrt(theta_fac);
                }
                rys_roots<NROOTS>(rr * theta * theta_fac, rw);
                // per primitive quartet: sum_n W_n (ij|kl)_n and the raised sums of i and k
                double e = 0.0, pi[3] = {0.0, 0.0, 0.0}, pk[3] = {0.0, 0.0, 0.0};
#pragma unroll 1
                for (int ir = 0; ir < NROOTS; ir++) {
                    const double rt = rw[2 * ir] * theta_fac;
                    const double wt = rw[2 * ir + 1] * sqrt_theta_fac;
                    const double rt_aa = rt * inv_aijkl;
                    const double rt_aij = rt_aa * akl, rt_akl = rt_aa * aij;
                    const double b10 = 0.5 * inv_aij * (1.0 - rt_aij);
                    const double b01 = 0.5 * inv_akl * (1.0 - rt_akl);
                    const double b00 = 0.5 * rt_aa;
                    double c0[3], cp[3];
#pragma unroll
                    for (int d = 0; d < 3; d++) {
                        c0[d] = fma(rjri[d], aj_aij, -rt_aij * Rpq[d]);
                        cp[d] = fma(rlrk[d], al_akl, rt_akl * Rpq[d]);
                    }
                    double g[3 * GS];
                    if constexpr (SMALL) fill_g_small<LI + 1, LJ, LK + 1, LL>(g, ckcl, gy0, wt, c0, cp, b10, b01, b00, rjri, rlrk);
                    else fill_g_large<LI + 1, LJ, LK + 1, LL>(g, ckcl, gy0, wt, c0, cp, b10, b01, b00, rjri, rlrk);
#pragma unroll U
                    for (int i = 0; i < NFI; i++)
#pragma unroll U
                    for (int j = 0; j < NFJ; j++)
#pragma unroll U
                    for (int k = 0; k < NFK; k++)
#pragma unroll U
                    for (int l = 0; l < NFL; l++) {
                        const int ix = CART_X[LI][i], iy = CART_Y[LI][i], iz = CART_Z[LI][i];
                        const int jx = CART_X[LJ][j], jy = CART_Y[LJ][j], jz = CART_Z[LJ][j];
                        const int kx = CART_X[LK][k], ky = CART_Y[LK][k], kz = CART_Z[LK][k];
                        const int ax = ix + jx * DJ + kx * DK + CART_X[LL][l] * DL;
                        const int ay = iy + jy * DJ + ky * DK + CART_Y[LL][l] * DL;
                        const int az = iz + jz * DJ + kz * DK + CART_Z[LL][l] * DL;
                        const double* __restrict__ gx = g;
                        const double* __restrict__ gyv = g + GS;
                        const double* __restrict__ gz = g + 2 * GS;
                        double wn;
                        if constexpr (SMALL) wn = w[((i * NFJ + j) * NFK + k) * NFL + l];
                        else wn = grad_weight<NSPIN>(a, i0 + i, j0 + j, k0 + k, l0 + l);
                        const double x = gx[ax], y = gyv[ay], z = gz[az];
                        const double wyz = wn * y * z, wxz = wn * x * z, wxy = wn * x * y;
                        e = fma(wyz, x, e);
                        pi[0] = fma(wyz, gx[ax + 1], pi[0]);
                        pi[1] = fma(wxz, gyv[ay + 1], pi[1]);
                        pi[2] = fma(wxy, gz[az + 1], pi[2]);
                        pk[0] = fma(wyz, gx[ax + DK], pk[0]);
                        pk[1] = fma(wxz, gyv[ay + DK], pk[1]);
                        pk[2] = fma(wxy, gz[az + DK], pk[2]);
                        if (ix > 0) mi[0] = fma(ix * wyz, gx[ax - 1], mi[0]);
                        if (iy > 0) mi[1] = fma(iy * wxz, gyv[ay - 1], mi[1]);
                        if (iz > 0) mi[2] = fma(iz * wxy, gz[az - 1], mi[2]);
                        if (jx > 0) mj[0] = fma(jx * wyz, gx[ax - DJ], mj[0]);
                        if (jy > 0) mj[1] = fma(jy * wxz, gyv[ay - DJ], mj[1]);
                        if (jz > 0) mj[2] = fma(jz * wxy, gz[az - DJ], mj[2]);
                        if (kx > 0) mk[0] = fma(kx * wyz, gx[ax - DK], mk[0]);
                        if (ky > 0) mk[1] = fma(ky * wxz, gyv[ay - DK], mk[1]);
                        if (kz > 0) mk[2] = fma(kz * wxy, gz[az - DK], mk[2]);
                    }
                }
                const double ai2 = 2.0 * cei.y, aj2 = 2.0 * cej.y, ak2 = 2.0 * cek.y;
#pragma unroll
                for (int d = 0; d < 3; d++) {
                    gi[d] = fma(ai2, pi[d], gi[d]);
                    gj[d] = fma(aj2, fma(-rjri[d], e, pi[d]), gj[d]);
                    gk[d] = fma(ak2, pk[d], gk[d]);
                }
            }
        }
        if (live) {
#pragma unroll
            for (int d = 0; d < 3; d++) {
                const double vi = gi[d] - mi[d], vj = gj[d] - mj[d], vk = gk[d] - mk[d];
                atomicAdd(a.gshell + 3 * ish + d, vi);
                atomicAdd(a.gshell + 3 * jsh + d, vj);
                atomicAdd(a.gshell + 3 * ksh + d, vk);
                atomicAdd(a.gshell + 3 * lsh + d, -((vi + vj) + vk));
            }
        }
    }
}

// Launchers, one translation unit per bra class (jk_grad_inst.cu).  Same class order as jk_launch:
// li >= lj, li >= lk, lk >= ll.  nspin: 1 (one density) or 2 (spin-unrestricted).
#define JQC_GRAD_DECL(I, J) \
    cudaError_t jk_grad_launch_##I##_##J(int lk, int ll, int nspin, const GradArgs& a, int nsm, cudaStream_t st);
JQC_GRAD_DECL(0, 0)
JQC_GRAD_DECL(1, 0) JQC_GRAD_DECL(1, 1)
JQC_GRAD_DECL(2, 0) JQC_GRAD_DECL(2, 1) JQC_GRAD_DECL(2, 2)
JQC_GRAD_DECL(3, 0) JQC_GRAD_DECL(3, 1) JQC_GRAD_DECL(3, 2) JQC_GRAD_DECL(3, 3)
JQC_GRAD_DECL(4, 0) JQC_GRAD_DECL(4, 1) JQC_GRAD_DECL(4, 2) JQC_GRAD_DECL(4, 3) JQC_GRAD_DECL(4, 4)
#undef JQC_GRAD_DECL

inline cudaError_t jk_grad_launch(int li, int lj, int lk, int ll, int nspin, const GradArgs& a, int nsm, cudaStream_t st)
{
#define JQC_CALL(I, J) if (li == I && lj == J) return jk_grad_launch_##I##_##J(lk, ll, nspin, a, nsm, st);
    JQC_CALL(0, 0)
    JQC_CALL(1, 0) JQC_CALL(1, 1)
    JQC_CALL(2, 0) JQC_CALL(2, 1) JQC_CALL(2, 2)
    JQC_CALL(3, 0) JQC_CALL(3, 1) JQC_CALL(3, 2) JQC_CALL(3, 3)
    JQC_CALL(4, 0) JQC_CALL(4, 1) JQC_CALL(4, 2) JQC_CALL(4, 3) JQC_CALL(4, 4)
#undef JQC_CALL
    return cudaErrorInvalidValue;
}

}  // namespace jqc
