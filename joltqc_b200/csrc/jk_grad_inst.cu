// One translation unit per bra class (JQC_LI >= JQC_LJ), compiled with -DJQC_LI=.. -DJQC_LJ=..
// Instantiates the J/K energy-gradient kernel (jk_grad.cuh) for every ket class lk <= li, ll <= lk,
// one density (NSPIN = 1) and two spin densities (NSPIN = 2), and exports one launcher.
#include <atomic>

#include "jk_grad.cuh"

namespace jqc {

// occupancy per device ordinal, computed on first use (as in jk_inst.cu)
constexpr int JQC_GRAD_MAX_DEVICES = 64;

template <int LK, int LL, int NSPIN>
static cudaError_t grad_launch_one(const GradArgs& a, int nsm, cudaStream_t st)
{
    constexpr bool SMALL = GradShape<JQC_LI, JQC_LJ, LK, LL>::SMALL;
    constexpr int NT = 128;
    auto kern = jk_grad_kernel<JQC_LI, JQC_LJ, LK, LL, SMALL, NT, NSPIN>;
    static std::atomic<int> cache[JQC_GRAD_MAX_DEVICES];
    int dev = 0;
    cudaError_t e = cudaGetDevice(&dev);
    if (e != cudaSuccess) return e;
    if (dev < 0 || dev >= JQC_GRAD_MAX_DEVICES) return cudaErrorInvalidDevice;
    int nb = cache[dev].load(std::memory_order_acquire);
    if (nb == 0) {
        e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nb, kern, NT, 0);
        if (e != cudaSuccess) return e;
        nb = nb > 0 ? nb : 1;
        cache[dev].store(nb, std::memory_order_release);
    }
    kern<<<nsm * nb, NT, 0, st>>>(a);
    return cudaGetLastError();
}

#define JQC_CAT_(a, b, c) a##b##_##c
#define JQC_CAT(a, b, c) JQC_CAT_(a, b, c)

// (templated on a dummy so that the discarded `if constexpr` branches are not instantiated)
template <int Z>
static cudaError_t grad_dispatch(int lk, int ll, int nspin, const GradArgs& a, int nsm, cudaStream_t st)
{
#define CASE(K, L)                                                                  \
    if constexpr (K + Z <= JQC_LI && L <= K) {                                      \
        if (lk == K && ll == L)                                                     \
            return nspin == 1 ? grad_launch_one<K, L, 1>(a, nsm, st) : grad_launch_one<K, L, 2>(a, nsm, st); \
    }
    CASE(0, 0)
    CASE(1, 0) CASE(1, 1)
    CASE(2, 0) CASE(2, 1) CASE(2, 2)
    CASE(3, 0) CASE(3, 1) CASE(3, 2) CASE(3, 3)
    CASE(4, 0) CASE(4, 1) CASE(4, 2) CASE(4, 3) CASE(4, 4)
#undef CASE
    return cudaErrorInvalidValue;
}

cudaError_t JQC_CAT(jk_grad_launch_, JQC_LI, JQC_LJ)(int lk, int ll, int nspin, const GradArgs& a, int nsm, cudaStream_t st)
{
    if (nspin != 1 && nspin != 2) return cudaErrorInvalidValue;
    return grad_dispatch<0>(lk, ll, nspin, a, nsm, st);
}

}  // namespace jqc
