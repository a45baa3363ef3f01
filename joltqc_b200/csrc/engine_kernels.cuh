// Helper kernels of the J/K engine: density pooling, task generation, AO transforms and the
// on-device Schwarz matrix.  Each cites the reference routine it stands in for.
#pragma once
#include <math_constants.h>

#include "jqc_common.cuh"

namespace jqc {

// ------------------------------------------------------------------ density pooling
// dm_cond[I,J] = max_b max_{mu in I, nu in J} |float(D_b[mu,nu])|  (reference:
// max_block_pooling, jqc/backend/linalg_helper.py:125-211, on the fp32 copy jk.py:172-173).
// One warp per row of shell blocks: lanes sweep the columns of the AO rows coalesced.
__global__ void dm_pool_kernel(const double* __restrict__ dm, int n_dm, int nao, int nbas,
                               const int* __restrict__ ao_loc, const int* __restrict__ ao2shell,
                               float* __restrict__ cond)
{
    const int I = blockIdx.x;
    const int r0 = ao_loc[I], r1 = ao_loc[I + 1];
    extern __shared__ float smax[];   // nbas floats
    for (int J = threadIdx.x; J < nbas; J += blockDim.x) smax[J] = 0.f;
    __syncthreads();
    const size_t nao2 = (size_t)nao * nao;
    for (int b = 0; b < n_dm; b++)
        for (int r = r0; r < r1; r++) {
            const double* row = dm + b * nao2 + (size_t)r * nao;
            for (int c = threadIdx.x; c < nao; c += blockDim.x) {
                const float v = fabsf((float)row[c]);
                // non-negative floats order like ints
                atomicMax(reinterpret_cast<int*>(&smax[ao2shell[c]]), __float_as_int(v));
            }
        }
    __syncthreads();
    for (int J = threadIdx.x; J < nbas; J += blockDim.x) cond[(size_t)I * nbas + J] = smax[J];
}

// log_dm_cond = log(dm_cond (+ transpose if hermi == 0)) in float32 and its global maximum
// (jk.py:179-184).  log_max is an ordered-int cell initialised to float_to_ordered(-inf).
__global__ void dm_log_kernel(const float* __restrict__ cond, int nbas, int hermi, float* __restrict__ logc,
                              int* __restrict__ log_max_ordered)
{
    const int J = blockIdx.y * blockDim.x + threadIdx.x;
    const int I = blockIdx.x;
    float lg = -CUDART_INF_F;
    if (J < nbas) {
        float v = cond[(size_t)I * nbas + J];
        if (hermi == 0) v += cond[(size_t)J * nbas + I];
        lg = logf(v);
        logc[(size_t)I * nbas + J] = lg;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) lg = fmaxf(lg, __shfl_xor_sync(0xffffffffu, lg, o));
    if ((threadIdx.x & 31) == 0) atomicMax(log_max_ordered, float_to_ordered(lg));
}

// ------------------------------------------------------------------ tile tables
// tile_q[ti*nt + tj] = max over the 4x4 shell tile of q (make_tile_pairs, jk.py:394)
__global__ void tile_max_kernel(const float* __restrict__ q, int nbas, float* __restrict__ tile_q)
{
    const int nt = nbas / TILE;
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nt * nt) return;
    const int ti = t / nt, tj = t - ti * nt;
    float m = -CUDART_INF_F;
#pragma unroll
    for (int a = 0; a < TILE; a++) {
        const float4 v = *reinterpret_cast<const float4*>(q + (size_t)(ti * TILE + a) * nbas + tj * TILE);
        m = fmaxf(m, fmaxf(fmaxf(v.x, v.y), fmaxf(v.z, v.w)));
    }
    tile_q[t] = m;
}

// Number of leading entries of each q-descending tile list that pass the pair cutoff
// log(1e-13) - log_max_dm (jk.py:185-187, 412).  One thread per group pair.
__global__ void active_tiles_kernel(const float* __restrict__ list_q, const int* __restrict__ list_off, int npairs,
                                    const int* __restrict__ log_max_ordered, int* __restrict__ n_active)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npairs) return;
    const double cutoff = log(1e-13) - (double)ordered_to_float(*log_max_ordered);
    int lo = list_off[p], hi = list_off[p + 1];
    const int base = lo;
    while (lo < hi) {   // first index whose q <= cutoff
        const int mid = (lo + hi) >> 1;
        if ((double)list_q[mid] > cutoff) lo = mid + 1; else hi = mid;
    }
    n_active[p] = lo - base;
}

// The same count for the energy-gradient screen, whose density factor is quadratic: the pair cutoff
// is log(1e-13) - 2 log_max_dm.
__global__ void active_tiles_grad_kernel(const float* __restrict__ list_q, const int* __restrict__ list_off, int npairs,
                                         const int* __restrict__ log_max_ordered, int* __restrict__ n_active)
{
    const int p = blockIdx.x * blockDim.x + threadIdx.x;
    if (p >= npairs) return;
    const double cutoff = log(1e-13) - 2.0 * (double)ordered_to_float(*log_max_ordered);
    int lo = list_off[p], hi = list_off[p + 1];
    const int base = lo;
    while (lo < hi) {
        const int mid = (lo + hi) >> 1;
        if ((double)list_q[mid] > cutoff) lo = mid + 1; else hi = mid;
    }
    n_active[p] = lo - base;
}

// ------------------------------------------------------------------ task generation
struct ScreenArgs {
    int nbas;
    const float* __restrict__ q;
    const float* __restrict__ logd;
    const float* __restrict__ logd_j;    // GRAD only: pooled log density of the J term (logd for one density)
    const int* __restrict__ log_max_ordered;
    const int* __restrict__ tiles_ij;    // tile ids ti*nt+tj, q-descending
    const int* __restrict__ tiles_kl;
    const float* __restrict__ tileq_kl;  // tile max q aligned with tiles_kl
    const int* __restrict__ nact_ij;     // device counts of active tiles in each list
    const int* __restrict__ nact_kl;
    int ij_begin, ij_count;              // chunk of this rank's slots: list index = shard_entry(ij_begin + s, rank, world)
    int kl_begin, kl_count;
    int rank, world;
    float cutoff;                        // log(cutoff_fp32): evaluate above this
    int do_j, do_k;
    ushort4* __restrict__ queue;
    unsigned* __restrict__ counter;          // queue entries written by this chunk
    unsigned long long* __restrict__ qcount; // quartets that passed (accounting)
    int tile_mode;                           // 1: emit (i, j, k-tile, l-tile, mask16) records for jk_tile16
};

// Thread = (one (i,j) shell pair of an ij tile) x (one kl tile): 16 quartet tests in the
// reference's canonical order and float32 log-domain criterion
// (jqc/backend/jk/screen_jk_tasks.cu:196-261), compacted per warp with one atomic.
// A warp holds 32 kl tiles for a single (i,j), so its output run shares i and j.
// GRAD selects the screen of the J/K energy gradient, whose weights are products of two density
// blocks: q_ij + q_kl + max(dJ_ij + dJ_kl [J], d_ik + d_jl, d_il + d_jk [K]) > cutoff, with the tile
// prefilter on 2 log max|D| (flat quartet records only).  dJ (logd_j) is the pooled density of the J
// term: logd itself for one density, the pooled Da + Db for two spin densities, where logd pools
// max_s |Ds| and log max|D| is the larger of the two maxima.
template <bool GRAD>
__global__ void __launch_bounds__(256) screen_tasks_kernel(const ScreenArgs s)
{
    const int nbas = s.nbas, nt = nbas / TILE;
    const int lane = threadIdx.x;
    const int kl_slot = blockIdx.x * 32 + lane;
    const int ij_slot = blockIdx.y * 8 + threadIdx.y;
    const int ij_idx = (int)shard_entry((unsigned)(s.ij_begin + (ij_slot >> 4)), s.rank, s.world);
    const int pair = ij_slot & 15;
    bool active = (ij_slot >> 4) < s.ij_count && ij_idx < *s.nact_ij && kl_slot < s.kl_count &&
                  (s.kl_begin + kl_slot) < *s.nact_kl;
    int ish = 0, jsh = 0, tk = 0, tl = 0;
    float q_ij = 0.f;
    const float log_max = fmaxf(ordered_to_float(*s.log_max_ordered), -36.8f);
    if (active) {
        const int tij = s.tiles_ij[ij_idx];
        const int ti = tij / nt, tj = tij - ti * nt;
        ish = ti * TILE + (pair >> 2);
        jsh = tj * TILE + (pair & 3);
        const int tkl = s.tiles_kl[s.kl_begin + kl_slot];
        tk = tkl / nt;
        tl = tkl - tk * nt;
        q_ij = s.q[(size_t)ish * nbas + jsh];
        active = ish >= jsh && tk * TILE <= ish &&
                 (q_ij + s.tileq_kl[s.kl_begin + kl_slot] + (GRAD ? 2.f * log_max : log_max) > s.cutoff);
    }
    unsigned mask = 0;
    if (active) {
        const int ksh0 = tk * TILE, lsh0 = tl * TILE;
        const float4 d_ik = *reinterpret_cast<const float4*>(s.logd + (size_t)ish * nbas + ksh0);
        const float4 d_jk = *reinterpret_cast<const float4*>(s.logd + (size_t)jsh * nbas + ksh0);
        const float4 d_il = *reinterpret_cast<const float4*>(s.logd + (size_t)ish * nbas + lsh0);
        const float4 d_jl = *reinterpret_cast<const float4*>(s.logd + (size_t)jsh * nbas + lsh0);
        const float dik[4] = {d_ik.x, d_ik.y, d_ik.z, d_ik.w}, djk[4] = {d_jk.x, d_jk.y, d_jk.z, d_jk.w};
        const float dil[4] = {d_il.x, d_il.y, d_il.z, d_il.w}, djl[4] = {d_jl.x, d_jl.y, d_jl.z, d_jl.w};
        const float* __restrict__ logd_j = GRAD ? s.logd_j : s.logd;
        const float d_ij = logd_j[(size_t)ish * nbas + jsh];
        const long long bas_ij = (long long)ish * nbas + jsh;
#pragma unroll
        for (int k = 0; k < TILE; k++) {
            const int ksh = ksh0 + k;
            const float4 qk = *reinterpret_cast<const float4*>(s.q + (size_t)ksh * nbas + lsh0);
            const float4 dk = *reinterpret_cast<const float4*>(logd_j + (size_t)ksh * nbas + lsh0);
            const float qkl[4] = {qk.x, qk.y, qk.z, qk.w}, dkl[4] = {dk.x, dk.y, dk.z, dk.w};
#pragma unroll
            for (int l = 0; l < TILE; l++) {
                const int lsh = lsh0 + l;
                if (ksh > ish || lsh > ksh || bas_ij < (long long)ksh * nbas + lsh) continue;
                const float q_ijkl = q_ij + qkl[l];
                if constexpr (GRAD) {
                    float d_large = -73.6f;
                    if (s.do_j) d_large = fmaxf(d_large, d_ij + dkl[l]);
                    if (s.do_k) {
                        d_large = fmaxf(d_large, dik[k] + djl[l]);
                        d_large = fmaxf(d_large, dil[l] + djk[k]);
                    }
                    const float dq = q_ijkl + d_large;
                    if (dq > s.cutoff) mask |= 1u << (k * TILE + l);
                } else {
                    float d_large = -36.8f;
                    if (s.do_k) {
                        d_large = fmaxf(d_large, dik[k]);
                        d_large = fmaxf(d_large, djk[k]);
                        d_large = fmaxf(d_large, dil[l]);
                        d_large = fmaxf(d_large, djl[l]);
                    }
                    if (s.do_j) {
                        d_large = fmaxf(d_large, d_ij);
                        d_large = fmaxf(d_large, dkl[l]);
                    }
                    const float dq = q_ijkl + d_large;
                    if (dq > s.cutoff) mask |= 1u << (k * TILE + l);
                }
            }
        }
    }
    const int cnt = __popc(mask);
    int incl = cnt;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const int n = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += n;
    }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    if (total == 0) return;
    if (lane == 31) atomicAdd(s.qcount, (unsigned long long)total);
    if (!GRAD && s.tile_mode) {
        // one 16-byte record per thread with survivors
        const unsigned has = __ballot_sync(0xffffffffu, mask != 0);
        unsigned base = 0;
        if (lane == 0) base = atomicAdd(s.counter, (unsigned)__popc(has));
        base = __shfl_sync(0xffffffffu, base, 0);
        if (mask) {
            uint4* q = reinterpret_cast<uint4*>(s.queue);
            q[base + __popc(has & ((1u << lane) - 1u))] =
                make_uint4((unsigned)ish | ((unsigned)jsh << 16), (unsigned)tk | ((unsigned)tl << 16), mask, 0u);
        }
        return;
    }
    unsigned base = 0;
    if (lane == 31) base = atomicAdd(s.counter, (unsigned)total);
    base = __shfl_sync(0xffffffffu, base, 31);
    unsigned pos = base + incl - cnt;
    while (mask) {
        const int b = __ffs(mask) - 1;
        mask &= mask - 1;
        s.queue[pos++] = make_ushort4((unsigned short)ish, (unsigned short)jsh,
                                      (unsigned short)(tk * TILE + (b >> 2)), (unsigned short)(tl * TILE + (b & 3)));
    }
}

// ------------------------------------------------------------------ energy gradient
// Dt = Da + Db of the spin-unrestricted gradient (kernel-side densities, n = nao^2 elements each)
__global__ void dm_spin_sum_kernel(const double* __restrict__ da, const double* __restrict__ db, double* __restrict__ dt,
                                   size_t n)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dt[i] = da[i] + db[i];
}

// Per-shell accumulator -> (natm, 3) gradient; shell_atom[s] = -1 for pads.  One thread per
// (atom, xyz), a fixed summation order (deterministic for a given accumulator).
__global__ void grad_shell_to_atom_kernel(const double* __restrict__ gshell, const int* __restrict__ shell_atom, int nbas,
                                          int natm, double* __restrict__ grad)
{
    const int t = blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= 3 * natm) return;
    const int atom = t / 3, d = t - 3 * atom;
    double s = 0.0;
    for (int sh = 0; sh < nbas; sh++)
        if (shell_atom[sh] == atom) s += gshell[3 * sh + d];
    grad[t] = s;
}

// ------------------------------------------------------------------ primitive-pair tables
// Static (geometry-only) data of every shell pair of a list, 8 doubles per primitive pair
// (first * n_second + second):  [a = a1 + a2, 1/a, a2/a, c1 c2 exp(-a1 a2/a |R12|^2), Px, Py, Pz, 0]
// with P = R1 + (a2/a)(R2 - R1).  The brick kernels read these instead of re-evaluating an exp and
// a division per primitive pair for every quartet (the reference recomputes them per quartet,
// 1q1t.cu:173-232; its pair algorithm stages the same quantities per block, pair_vj.cu:139-220).
__global__ void pair_prim_kernel(const double* __restrict__ basis, const ushort2* __restrict__ pairs, int n, int np1,
                                 int np2, double* __restrict__ out)
{
    const int npp = np1 * np2;
    const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= (long long)n * npp) return;
    const int e = (int)(idx / npp), pp = (int)(idx - (long long)e * npp);
    const int p1 = pp / np2, p2 = pp - p1 * np2;
    const ushort2 sh = pairs[e];
    const double* __restrict__ b1 = basis + sh.x * BASIS_STRIDE;
    const double* __restrict__ b2 = basis + sh.y * BASIS_STRIDE;
    const double dx = b2[0] - b1[0], dy = b2[1] - b1[1], dz = b2[2] - b1[2];
    const double rr = dx * dx + dy * dy + dz * dz;
    const double c1 = b1[4 + 2 * p1], a1 = b1[5 + 2 * p1], c2 = b2[4 + 2 * p2], a2 = b2[5 + 2 * p2];
    const double a = a1 + a2;
    const double inv_a = 1.0 / a;
    const double a2_a = a2 * inv_a;
    double* __restrict__ o = out + idx * 8;
    o[0] = a;
    o[1] = inv_a;
    o[2] = a2_a;
    o[3] = c1 * c2 * exp(-a1 * a2_a * rr);
    o[4] = fma(dx, a2_a, b1[0]);
    o[5] = fma(dy, a2_a, b1[1]);
    o[6] = fma(dz, a2_a, b1[2]);
    o[7] = 0.0;
}

// ------------------------------------------------------------------ AO transforms
struct XformTab {
    const double* __restrict__ c2s;   // concatenated (ncart x nmol) matrices, identity when the molecule is cartesian
    int off[LMAX + 1];                // offsets into c2s
    int nmol[LMAX + 1];               // 2l+1 or ncart
};

// kernel side <- molecule: D_k[mu,nu] = sum_mn C[c_mu,m] D_mol[P(mu)+m, P(nu)+n] C[c_nu,n]
// (dm_from_mol, basis.py:419-450; sph2cart.cu:335-362 / cart2cart cart2sph.py:241-307).
__global__ void dm_from_mol_kernel(const double* __restrict__ mol, int mol_nao, double* __restrict__ kern, int nao,
                                   const int* __restrict__ ao2shell, const int* __restrict__ ao_loc,
                                   const int* __restrict__ angs, const int* __restrict__ mol_off, XformTab t,
                                   int transpose_out)
{
    const int nu = blockIdx.y * blockDim.x + threadIdx.x;
    const int mu = blockIdx.x;
    if (nu >= nao) return;
    const size_t b = blockIdx.z;
    const int s1 = ao2shell[mu], s2 = ao2shell[nu];
    const int l1 = angs[s1], l2 = angs[s2];
    const int c1 = mu - ao_loc[s1], c2 = nu - ao_loc[s2];
    const int n1 = t.nmol[l1], n2 = t.nmol[l2];
    const double* C1 = t.c2s + t.off[l1] + c1 * n1;
    const double* C2 = t.c2s + t.off[l2] + c2 * n2;
    const double* src = mol + b * (size_t)mol_nao * mol_nao + (size_t)mol_off[s1] * mol_nao + mol_off[s2];
    double acc = 0.0;
    for (int m = 0; m < n1; m++) {
        const double a = C1[m];
        if (a == 0.0) continue;
        double r = 0.0;
        for (int n = 0; n < n2; n++) r = fma(C2[n], src[(size_t)m * mol_nao + n], r);
        acc = fma(a, r, acc);
    }
    double* dst = kern + b * (size_t)nao * nao;
    if (transpose_out) dst[(size_t)nu * nao + mu] = acc; else dst[(size_t)mu * nao + nu] = acc;
}

// molecule <- kernel side with the reference's post-processing folded into the read
// (jk.py:353-370) and the accumulation over split siblings done as a gather instead of
// atomics (dm_to_mol, basis.py:452-480; cart2sph.cu:273-300).
//   mode 0: plain            W = A[b]
//   mode 1: hermi=1 J        W = 2 (A[b] + A[b]^T)
//   mode 2: hermi=1 K        W = A[b] + A[b]^T
//   mode 3: hermi!=1 J       W = S + S^T,  S = A[b] + A[b+n]^T
//   mode 4: hermi!=1 K       W = A[b] + A[b+n]^T
__device__ __forceinline__ double post_read(const double* __restrict__ A, size_t nao, size_t b, size_t n, int mode,
                                            size_t r, size_t c)
{
    const size_t nao2 = nao * nao;
    const double* A0 = A + b * nao2;
    switch (mode) {
        case 0: return A0[r * nao + c];
        case 1: return 2.0 * (A0[r * nao + c] + A0[c * nao + r]);
        case 2: return A0[r * nao + c] + A0[c * nao + r];
        case 3: { const double* A1 = A + (b + n) * nao2;
                  return (A0[r * nao + c] + A1[c * nao + r]) + (A0[c * nao + r] + A1[r * nao + c]); }
        default: { const double* A1 = A + (b + n) * nao2; return A0[r * nao + c] + A1[c * nao + r]; }
    }
}

__global__ void dm_to_mol_kernel(const double* __restrict__ kern, int nao, int n, int mode, double* __restrict__ mol,
                                 int mol_nao, const int* __restrict__ molao_parent, const int* __restrict__ molao_m,
                                 const int* __restrict__ child_ptr, const int* __restrict__ child_list,
                                 const int* __restrict__ ao_loc, const int* __restrict__ angs, XformTab t)
{
    const int q = blockIdx.y * blockDim.x + threadIdx.x;
    const int p = blockIdx.x;
    if (q >= mol_nao) return;
    const size_t b = blockIdx.z;
    const int P = molao_parent[p], Q = molao_parent[q];
    const int m = molao_m[p], nn = molao_m[q];
    double acc = 0.0;
    for (int a = child_ptr[P]; a < child_ptr[P + 1]; a++) {
        const int s1 = child_list[a];
        const int l1 = angs[s1], nc1 = nf_of(l1), n1 = t.nmol[l1];
        const double* C1 = t.c2s + t.off[l1];
        for (int bb = child_ptr[Q]; bb < child_ptr[Q + 1]; bb++) {
            const int s2 = child_list[bb];
            const int l2 = angs[s2], nc2 = nf_of(l2), n2 = t.nmol[l2];
            const double* C2 = t.c2s + t.off[l2];
            for (int c1 = 0; c1 < nc1; c1++) {
                const double x = C1[c1 * n1 + m];
                if (x == 0.0) continue;
                double r = 0.0;
                for (int c2 = 0; c2 < nc2; c2++) {
                    const double y = C2[c2 * n2 + nn];
                    if (y != 0.0) r = fma(y, post_read(kern, nao, b, n, mode, ao_loc[s1] + c1, ao_loc[s2] + c2), r);
                }
                acc = fma(x, r, acc);
            }
        }
    }
    mol[b * (size_t)mol_nao * mol_nao + (size_t)p * mol_nao + q] = acc;
}

// ------------------------------------------------------------------ generic ERI (any l <= 4)
// Run-time-l evaluation of one cartesian block (ab|cd) into `out` (global scratch), used only
// by the one-off Schwarz matrix.  Same recurrences as the specialised kernels.
struct GenScratch {
    double t[3][2 * LMAX + 1][2 * LMAX + 1];
    double h[3][2 * LMAX + 1][LMAX + 1][2 * LMAX + 1];
    double g[3][LMAX + 1][LMAX + 1][LMAX + 1][LMAX + 1];
};

__device__ void rys_roots_rt(int nroots, double x, double* rw)
{
    switch (nroots) {
        case 1: rys_roots<1>(x, rw); break;
        case 2: rys_roots<2>(x, rw); break;
        case 3: rys_roots<3>(x, rw); break;
        case 4: rys_roots<4>(x, rw); break;
        case 5: rys_roots<5>(x, rw); break;
        case 6: rys_roots<6>(x, rw); break;
        case 7: rys_roots<7>(x, rw); break;
        case 8: rys_roots<8>(x, rw); break;
        default: rys_roots<9>(x, rw); break;
    }
}

__device__ void eri_generic(const double* __restrict__ basis, int ish, int jsh, int ksh, int lsh, int li, int lj,
                            int lk, int ll, int npi, int npj, int npk, int npl, double omega, double fac,
                            GenScratch* __restrict__ w, double* __restrict__ out)
{
    const double* bi = basis + ish * BASIS_STRIDE;
    const double* bj = basis + jsh * BASIS_STRIDE;
    const double* bk = basis + ksh * BASIS_STRIDE;
    const double* bl = basis + lsh * BASIS_STRIDE;
    const int lij = li + lj, lkl = lk + ll, nroots = (lij + lkl) / 2 + 1;
    const int nfi = nf_of(li), nfj = nf_of(lj), nfk = nf_of(lk), nfl = nf_of(ll);
    double rjri[3], rlrk[3], rr_ij = 0, rr_kl = 0;
    for (int d = 0; d < 3; d++) {
        rjri[d] = bj[d] - bi[d]; rr_ij += rjri[d] * rjri[d];
        rlrk[d] = bl[d] - bk[d]; rr_kl += rlrk[d] * rlrk[d];
    }
    const int n = nfi * nfj * nfk * nfl;
    for (int e = 0; e < n; e++) out[e] = 0.0;
    double rw[18];
    for (int kp = 0; kp < npk; kp++)
    for (int lp = 0; lp < npl; lp++) {
        const double ak = bk[5 + 2 * kp], al = bl[5 + 2 * lp];
        const double akl = ak + al, inv_akl = 1.0 / akl, al_akl = al * inv_akl;
        const double ckcl = bk[4 + 2 * kp] * bl[4 + 2 * lp] * exp(-ak * al_akl * rr_kl);
        for (int ip = 0; ip < npi; ip++)
        for (int jp = 0; jp < npj; jp++) {
            const double ai = bi[5 + 2 * ip], aj = bj[5 + 2 * jp];
            const double aij = ai + aj, inv_aij = 1.0 / aij, aj_aij = aj * inv_aij;
            const double cicj = fac * bi[4 + 2 * ip] * bj[4 + 2 * jp] * exp(-ai * aj_aij * rr_ij);
            double Rpq[3], rr = 0;
            for (int d = 0; d < 3; d++) {
                Rpq[d] = (rjri[d] * aj_aij + bi[d]) - (rlrk[d] * al_akl + bk[d]);
                rr += Rpq[d] * Rpq[d];
            }
            const double inv_aijkl = 1.0 / (aij + akl);
            const double theta = aij * akl * inv_aijkl;
            const double gy0 = cicj * inv_aij * inv_akl * sqrt(inv_aijkl);
            double theta_fac = 1.0, sqrt_theta_fac = 1.0;
            if (omega > 0.0) {
                theta_fac = omega * omega / (omega * omega + theta);
                sqrt_theta_fac = sqrt(theta_fac);
            }
            rys_roots_rt(nroots, rr * theta * theta_fac, rw);
            for (int ir = 0; ir < nroots; ir++) {
                const double rt = rw[2 * ir] * theta_fac, wt = rw[2 * ir + 1] * sqrt_theta_fac;
                const double rt_aa = rt * inv_aijkl, rt_aij = rt_aa * akl, rt_akl = rt_aa * aij;
                const double b10 = .5 * inv_aij * (1.0 - rt_aij), b01 = .5 * inv_akl * (1.0 - rt_akl), b00 = .5 * rt_aa;
                for (int d = 0; d < 3; d++) {
                    const double c0 = rjri[d] * aj_aij - rt_aij * Rpq[d];
                    const double cp = rlrk[d] * al_akl + rt_akl * Rpq[d];
                    w->t[d][0][0] = d == 0 ? ckcl : (d == 1 ? gy0 : wt);
                    for (int i = 0; i < lij; i++)
                        w->t[d][i + 1][0] = c0 * w->t[d][i][0] + (i > 0 ? i * b10 * w->t[d][i - 1][0] : 0.0);
                    for (int k = 0; k < lkl; k++)
                        for (int i = 0; i <= lij; i++) {
                            double v = cp * w->t[d][i][k];
                            if (k > 0) v += k * b01 * w->t[d][i][k - 1];
                            if (i > 0) v += i * b00 * w->t[d][i - 1][k];
                            w->t[d][i][k + 1] = v;
                        }
                    for (int k = 0; k <= lkl; k++) {
                        for (int i = 0; i <= lij; i++) w->h[d][i][0][k] = w->t[d][i][k];
                        for (int j = 0; j < lj; j++)
                            for (int i = 0; i <= lij - j - 1; i++)
                                w->h[d][i][j + 1][k] = w->h[d][i + 1][j][k] - rjri[d] * w->h[d][i][j][k];
                    }
                    for (int i = 0; i <= li; i++)
                        for (int j = 0; j <= lj; j++) {
                            // ket HRR in place on the t row (reused as scratch): v[k][l]
                            double v[2 * LMAX + 1][LMAX + 1];
                            for (int k = 0; k <= lkl; k++) v[k][0] = w->h[d][i][j][k];
                            for (int l = 0; l < ll; l++)
                                for (int k = 0; k <= lkl - l - 1; k++) v[k][l + 1] = v[k + 1][l] - rlrk[d] * v[k][l];
                            for (int k = 0; k <= lk; k++)
                                for (int l = 0; l <= ll; l++) w->g[d][i][j][k][l] = v[k][l];
                        }
                }
                double* o = out;
                for (int i = 0; i < nfi; i++)
                for (int j = 0; j < nfj; j++)
                for (int k = 0; k < nfk; k++)
                for (int l = 0; l < nfl; l++)
                    *o++ += w->g[0][CART_X[li][i]][CART_X[lj][j]][CART_X[lk][k]][CART_X[ll][l]] *
                            w->g[1][CART_Y[li][i]][CART_Y[lj][j]][CART_Y[lk][k]][CART_Y[ll][l]] *
                            w->g[2][CART_Z[li][i]][CART_Z[lj][j]][CART_Z[lk][k]][CART_Z[ll][l]];
            }
        }
    }
}

// q[i,j] = log(sqrt(max_ab |(ab|ab)|) + 1e-300) over cartesian or real-spherical components,
// float32, pads -100: the definition of libcint's CVHFnr_int2e_q_cond that the reference calls
// on the CPU (jqc/pyscf/basis.py:840-867, 237-239).  Grid-stride over shell pairs i >= j.
__global__ void q_cond_kernel(const double* __restrict__ basis, const int* __restrict__ angs,
                              const int* __restrict__ nprims, const unsigned char* __restrict__ pad, int nbas,
                              int cart, XformTab t, double omega, GenScratch* __restrict__ scratch,
                              double* __restrict__ blocks, int blk_stride, float* __restrict__ q)
{
    const int tid = blockIdx.x * blockDim.x + threadIdx.x;
    const long long npair = (long long)nbas * (nbas + 1) / 2;
    GenScratch* w = scratch + tid;
    double* blk = blocks + (size_t)tid * blk_stride;
    for (long long p = tid; p < npair; p += (long long)gridDim.x * blockDim.x) {
        int i = (int)((sqrt(8.0 * (double)p + 1.0) - 1.0) * 0.5);
        while ((long long)i * (i + 1) / 2 > p) i--;
        while ((long long)(i + 1) * (i + 2) / 2 <= p) i++;
        const int j = (int)(p - (long long)i * (i + 1) / 2);
        float val = -100.f;
        if (!pad[i] && !pad[j]) {
            const int li = angs[i], lj = angs[j];
            eri_generic(basis, i, j, i, j, li, lj, li, lj, nprims[i], nprims[j], nprims[i], nprims[j], omega, PI_FAC,
                        w, blk);
            const int nfi = nf_of(li), nfj = nf_of(lj);
            double m = 0.0;
            if (cart) {
                for (int a = 0; a < nfi; a++)
                    for (int b = 0; b < nfj; b++) m = fmax(m, fabs(blk[((a * nfj + b) * nfi + a) * nfj + b]));
            } else {
                const int di = 2 * li + 1, dj = 2 * lj + 1;
                const double* ci = t.c2s + t.off[li];
                const double* cj = t.c2s + t.off[lj];
                for (int ma = 0; ma < di; ma++)
                    for (int mb = 0; mb < dj; mb++) {
                        double e = 0.0;
                        for (int a = 0; a < nfi; a++) {
                            const double xa = ci[a * di + ma];
                            if (xa == 0.0) continue;
                            for (int b = 0; b < nfj; b++) {
                                const double xb = xa * cj[b * dj + mb];
                                if (xb == 0.0) continue;
                                for (int c = 0; c < nfi; c++) {
                                    const double xc = xb * ci[c * di + ma];
                                    if (xc == 0.0) continue;
                                    for (int d = 0; d < nfj; d++)
                                        e = fma(xc * cj[d * dj + mb], blk[((a * nfj + b) * nfi + c) * nfj + d], e);
                                }
                            }
                        }
                        m = fmax(m, fabs(e));
                    }
            }
            val = (float)log(sqrt(m) + 1e-300);
        }
        q[(size_t)i * nbas + j] = val;
        q[(size_t)j * nbas + i] = val;
    }
}

// ------------------------------------------------------------------ FP64 peak probe
// 8 independent DFMA chains per thread, all in registers: sustained FMA-pipe rate.
// float copy of the kernel-side density for the FP32-band launches (the reference keeps dms_fp32,
// jqc/pyscf/jk.py:197-199)
__global__ void to_float_kernel(const double* __restrict__ src, float* __restrict__ dst, size_t n)
{
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
        dst[i] = (float)src[i];
}

__global__ void fp64_probe_kernel(double* out, int iters, double a, double b)
{
    double x0 = threadIdx.x * 1e-9, x1 = x0 + 1, x2 = x0 + 2, x3 = x0 + 3, x4 = x0 + 4, x5 = x0 + 5, x6 = x0 + 6, x7 = x0 + 7;
    for (int i = 0; i < iters; i++) {
#pragma unroll
        for (int u = 0; u < 8; u++) {
            x0 = fma(x0, a, b); x1 = fma(x1, a, b); x2 = fma(x2, a, b); x3 = fma(x3, a, b);
            x4 = fma(x4, a, b); x5 = fma(x5, a, b); x6 = fma(x6, a, b); x7 = fma(x7, a, b);
        }
    }
    const double s = ((x0 + x1) + (x2 + x3)) + ((x4 + x5) + (x6 + x7));
    if (s == 123.456) out[0] = s;
}

}  // namespace jqc
