// joltqc_b200 J/K engine: host orchestration + C ABI (include/joltqc_b200.h).
//
// One engine = one shell table on one GPU.  A build enqueues, without any host
// synchronisation:  AO transform in -> density pooling -> per group quartet
// { task generation into a device queue -> Rys kernel reading the queue length from device
// memory } -> post-processing + AO transform out.  (The reference round-trips to the host
// after every task-generation launch, jqc/pyscf/jk.py:280, and re-allocates a 2 GiB queue
// per call, jk.py:207.)
#include <algorithm>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <map>
#include <memory>
#include <numeric>
#include <string>
#include <vector>

#include "../../include/joltqc_b200.h"
#include "engine_kernels.cuh"
#include "jk_brick.cuh"
#include "jk_grad.cuh"
#include "jk_launch.h"

using namespace jqc;

static thread_local std::string g_err;
static int fail(int code, const std::string& msg)
{
    g_err = msg;
    return code;
}
#define CU(call)                                                                                  \
    do {                                                                                          \
        cudaError_t e_ = (call);                                                                  \
        if (e_ != cudaSuccess)                                                                    \
            return fail(JQC_ECUDA, std::string(#call) + ": " + cudaGetErrorString(e_));           \
    } while (0)

namespace {

constexpr size_t QUEUE_CAP = size_t(1) << 27;   // ushort4 entries (1 GiB) at most, allocated on first use
constexpr int MAX_CHUNKS = 1 << 18;

template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    ~DevBuf() { if (p) cudaFree(p); }
    cudaError_t ensure(size_t count)
    {
        if (count <= n) return cudaSuccess;
        if (p) cudaFree(p);
        p = nullptr; n = 0;
        cudaError_t e = cudaMalloc(&p, count * sizeof(T));
        if (e == cudaSuccess) n = count;
        return e;
    }
    cudaError_t upload(const std::vector<T>& v)
    {
        cudaError_t e = ensure(std::max<size_t>(v.size(), 1));
        if (e != cudaSuccess) return e;
        return cudaMemcpy(p, v.data(), v.size() * sizeof(T), cudaMemcpyHostToDevice);
    }
};

struct QData {                    // per-omega Schwarz data
    DevBuf<float> q;              // nbas x nbas
    DevBuf<int> tiles;            // concatenated q-descending tile lists, one per group pair
    DevBuf<float> tiles_q;
    DevBuf<int> list_off;         // npairs + 1
    std::vector<int> h_list_off;
    // shell-pair lists of the brick kernel (jk_brick.cuh), one segment per group pair (ga >= gb):
    //   ket role: pairs ordered by (bucket of 32 shells of ga, q descending) -> 32 neighbours = one brick
    //   bra role: for every shell a of ga its partners b, q descending (CSR)
    DevBuf<ushort2> kl;
    DevBuf<float> kl_q, kl_tq;
    DevBuf<unsigned short> j_idx;
    DevBuf<float> j_q, j_tq;
    DevBuf<int> j_off;            // per group pair: (size of ga) + 1 offsets, absolute into j_idx
    std::vector<int> h_pair_off;  // npairs + 1: segment of each group pair in kl / j_idx
    std::vector<int> h_joff_off;  // npairs: start of each group pair's row offsets in j_off
    std::vector<float> h_qmax;    // npairs: largest q of the group pair
    // primitive-pair tables in ket-list and bra-list order (pair_prim_kernel), 8 doubles per primitive pair
    DevBuf<double> ket_tab, bra_tab;
    std::vector<size_t> h_tab_off;   // npairs: offset (doubles) of each group pair's segment in both tables
};

struct ChunkRec { int key; long long pw; bool fp32 = false; };   // class key, primitive weight, precision of a launch

}  // namespace

struct jqc_engine {
    int device = 0, nsm = 148;
    int nbas = 0, nao = 0, ngroups = 0, mol_nao = 0, mol_cart = 0, nt = 0, lmax = 0;
    std::vector<int> angs, nprims, ao_loc, goff, gl, gnp, mol_off;
    std::vector<uint8_t> pad;
    DevBuf<double> d_basis, d_c2s;
    DevBuf<int> d_angs, d_nprims, d_ao_loc, d_ao2shell, d_mol_off;
    DevBuf<unsigned char> d_pad;
    DevBuf<int> d_molao_parent, d_molao_m, d_child_ptr, d_child_list;
    XformTab xt{};
    std::map<double, std::unique_ptr<QData>> qcache;
    // per-call scratch
    DevBuf<double> d_dm, d_vjk, d_stage_in, d_stage_j, d_stage_k;
    DevBuf<float> d_cond, d_logd, d_dm32;
    DevBuf<int> d_logmax, d_nact;
    DevBuf<ushort4> d_queue;
    DevBuf<unsigned> d_counters;
    DevBuf<unsigned long long> d_qcounts;
    // energy gradient (jqc_jk_energy_grad): own task counters, so that the accounting of the last J/K
    // build stays readable, plus the per-shell accumulator and the shell -> atom map
    DevBuf<unsigned> d_gcounters;
    DevBuf<unsigned long long> d_gqcounts;
    DevBuf<double> d_gshell;
    DevBuf<int> d_gatom;
    DevBuf<float> d_glogdj;   // pooled log density of the J term (Da + Db) of the spin-unrestricted gradient
    int rank = 0, world = 1;
    // task format for blocks of <= 81 integrals: 0 flat quartets (default), 1 4x4 tile records.
    // Both were measured in round 1 (profiles/README.md); JQC_SMALL_TILES=1 selects the tile kernel.
    int small_tiles = 0;
    // brick kernel (jk_brick.cuh) for the classes of <= 108 integrals and one density matrix;
    // JQC_BRICK=0 falls back to the quartet-list kernels (kept as the cross-check of the tests)
    int use_brick = 1;
    int use_bwarp = 1;          // brick-scheduled multi-lane kernel (jk_bwarp.cuh) for the larger classes
    int brick_ichunk = 8;
    // chunking of the quartet-list path; JQC_QUEUE_CAP / JQC_KL_CHUNK shrink them so that small test
    // molecules exercise the multi-chunk loops
    size_t queue_cap = QUEUE_CAP;
    int kl_chunk_max = 2048;
    // brick launches need no queue: they go round-robin to auxiliary streams so that the tail of one
    // launch overlaps the start of the next (and the quartet-list launches of the main stream)
    static constexpr int NAUX = 3;
    cudaStream_t aux[NAUX] = {nullptr, nullptr, nullptr};
    cudaEvent_t ev_fork = nullptr, ev_join[NAUX] = {nullptr, nullptr, nullptr};
    int use_aux = 1;
    int use_fp32 = 1;
    // state of the last build
    int last_n = 0, last_neff = 0, last_hermi = 1, last_j = 0, last_k = 0, launches = 0;
    bool built = false, profiling = false;
    std::vector<ChunkRec> chunks;
    long long band_n[2] = {0, 0};   // quartets evaluated by the FP64 / FP32 kernels in the last build
    float band_ms[2] = {0.f, 0.f};
    std::vector<cudaEvent_t> ev;
    std::vector<float> class_ms = std::vector<float>(625, 0.f);
    int npairs() const { return ngroups * (ngroups + 1) / 2; }
    static int pair_id(int gi, int gj) { return gi * (gi + 1) / 2 + gj; }
};

// ---------------------------------------------------------------------------------------
extern "C" const char* jqc_last_error(void) { return g_err.c_str(); }

extern "C" int jqc_engine_create(const jqc_basis_desc* d, int device, jqc_engine** out)
{
    if (!d || !out) return fail(JQC_EINVAL, "null argument");
    // 56 K shells: ushort shell indices and one float per shell of dynamic shared memory in dm_pool_kernel
    if (d->nbas <= 0 || d->nbas % JQC_TILE || d->nbas > 56 * 1024)
        return fail(JQC_EINVAL, "nbas must be a positive multiple of 4 and <= 57344");
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(JQC_ECUDA, "no CUDA device: joltqc_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(JQC_EINVAL, "bad device ordinal");
    CU(cudaSetDevice(device));
    std::unique_ptr<jqc_engine> e(new jqc_engine);
    e->device = device;
    if (const char* m = getenv("JQC_SMALL_TILES")) e->small_tiles = atoi(m) != 0;
    if (const char* m = getenv("JQC_BRICK")) e->use_brick = atoi(m) != 0;
    if (const char* m = getenv("JQC_BWARP")) e->use_bwarp = atoi(m);   // 0 off, 1 measured table, 2 every supported class
    if (const char* m = getenv("JQC_BRICK_ICHUNK")) e->brick_ichunk = std::max(1, atoi(m));
    if (const char* m = getenv("JQC_AUX_STREAMS")) e->use_aux = atoi(m) != 0;
    if (const char* m = getenv("JQC_FP32")) e->use_fp32 = atoi(m) != 0;     // 0: evaluate the FP32 band in FP64
    if (const char* m = getenv("JQC_QUEUE_CAP")) e->queue_cap = std::min<size_t>(QUEUE_CAP, std::max<size_t>(256, (size_t)atoll(m)));
    if (const char* m = getenv("JQC_KL_CHUNK")) e->kl_chunk_max = std::max(1, atoi(m));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    e->nsm = prop.multiProcessorCount;
    e->nbas = d->nbas;
    e->ngroups = d->ngroups;
    e->mol_nao = d->mol_nao;
    e->mol_cart = d->mol_cart;
    e->nt = d->nbas / JQC_TILE;
    e->angs.assign(d->angs, d->angs + d->nbas);
    e->nprims.assign(d->nprims, d->nprims + d->nbas);
    e->ao_loc.assign(d->ao_loc, d->ao_loc + d->nbas + 1);
    e->pad.assign(d->pad, d->pad + d->nbas);
    e->goff.assign(d->group_offset, d->group_offset + d->ngroups + 1);
    e->mol_off.assign(d->mol_ao_offset, d->mol_ao_offset + d->nbas);
    e->nao = e->ao_loc[d->nbas];
    for (int g = 0; g < d->ngroups; g++) {
        const int s0 = e->goff[g], s1 = e->goff[g + 1];
        if (s0 % JQC_TILE || s1 <= s0 || s1 > d->nbas) return fail(JQC_EINVAL, "group offsets must be increasing multiples of 4");
        e->gl.push_back(e->angs[s0]);
        e->gnp.push_back(e->nprims[s0]);
        for (int s = s0; s < s1; s++)
            if (e->angs[s] != e->angs[s0] || e->nprims[s] != e->nprims[s0])
                return fail(JQC_EINVAL, "shells of one group must share (l, nprim)");
        if (g > 0 && e->gl[g] < e->gl[g - 1]) return fail(JQC_EINVAL, "groups must be ordered by l ascending");
    }
    for (int s = 0; s < d->nbas; s++) {
        if (e->angs[s] < 0 || e->angs[s] > JQC_LMAX) return fail(JQC_EINVAL, "angular momentum above 4");
        if (e->nprims[s] < 1 || e->nprims[s] > JQC_NPRIM_MAX) return fail(JQC_EINVAL, "nprim must be 1..3");
        e->lmax = std::max(e->lmax, e->angs[s]);
    }
    // uploads
    std::vector<double> rec(d->records, d->records + (size_t)d->nbas * JQC_BASIS_STRIDE);
    CU(e->d_basis.upload(rec));
    CU(e->d_angs.upload(e->angs));
    CU(e->d_nprims.upload(e->nprims));
    CU(e->d_ao_loc.upload(e->ao_loc));
    CU(e->d_mol_off.upload(e->mol_off));
    std::vector<unsigned char> padv(e->pad.begin(), e->pad.end());
    CU(e->d_pad.upload(padv));
    std::vector<int> ao2shell(std::max(e->nao, 1));
    for (int s = 0; s < d->nbas; s++)
        for (int a = e->ao_loc[s]; a < e->ao_loc[s + 1]; a++) ao2shell[a] = s;
    CU(e->d_ao2shell.upload(ao2shell));
    // transform tables
    std::vector<double> c2s;
    int off_in = 0;
    for (int l = 0; l <= JQC_LMAX; l++) {
        const int nc = (l + 1) * (l + 2) / 2, ns = 2 * l + 1;
        e->xt.off[l] = (int)c2s.size();
        if (d->mol_cart) {
            e->xt.nmol[l] = nc;
            for (int a = 0; a < nc; a++)
                for (int b = 0; b < nc; b++) c2s.push_back(a == b ? 1.0 : 0.0);
        } else {
            if (!d->c2s) return fail(JQC_EINVAL, "c2s matrices are required for a spherical molecule");
            e->xt.nmol[l] = ns;
            c2s.insert(c2s.end(), d->c2s + off_in, d->c2s + off_in + nc * ns);
        }
        off_in += nc * ns;
    }
    CU(e->d_c2s.upload(c2s));
    e->xt.c2s = e->d_c2s.p;
    // molecule AO -> (parent id, component) and parent -> children
    std::map<int, int> parent_of_off;   // mol offset -> parent id
    std::vector<int> shell_parent(d->nbas, -1);
    for (int s = 0; s < d->nbas; s++) {
        if (e->pad[s]) continue;
        if (e->mol_off[s] < 0) return fail(JQC_EINVAL, "non-pad shell without molecular AO offset");
        auto it = parent_of_off.find(e->mol_off[s]);
        if (it == parent_of_off.end()) it = parent_of_off.emplace(e->mol_off[s], (int)parent_of_off.size()).first;
        shell_parent[s] = it->second;
    }
    const int nparent = (int)parent_of_off.size();
    std::vector<std::vector<int>> children(nparent);
    for (int s = 0; s < d->nbas; s++)
        if (shell_parent[s] >= 0) children[shell_parent[s]].push_back(s);
    std::vector<int> molao_parent(std::max(e->mol_nao, 1), -1), molao_m(std::max(e->mol_nao, 1), 0), cptr(nparent + 1, 0), clist;
    for (auto& kv : parent_of_off) {
        const int P = kv.second, l = e->angs[children[P][0]];
        const int nm = e->xt.nmol[l];
        if (kv.first + nm > e->mol_nao) return fail(JQC_EINVAL, "molecular AO offset out of range");
        for (int m = 0; m < nm; m++) { molao_parent[kv.first + m] = P; molao_m[kv.first + m] = m; }
    }
    for (int a = 0; a < e->mol_nao; a++)
        if (molao_parent[a] < 0) return fail(JQC_EINVAL, "molecular AO not covered by any shell");
    for (int P = 0; P < nparent; P++) {
        cptr[P + 1] = cptr[P] + (int)children[P].size();
        clist.insert(clist.end(), children[P].begin(), children[P].end());
    }
    CU(e->d_molao_parent.upload(molao_parent));
    CU(e->d_molao_m.upload(molao_m));
    CU(e->d_child_ptr.upload(cptr));
    CU(e->d_child_list.upload(clist));
    if ((size_t)d->nbas * sizeof(float) > 48 * 1024)   // dm_pool_kernel keeps one row of shell maxima in shared memory
        CU(cudaFuncSetAttribute(dm_pool_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(d->nbas * sizeof(float))));
    for (int i = 0; i < jqc_engine::NAUX; i++) {
        CU(cudaStreamCreateWithFlags(&e->aux[i], cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&e->ev_join[i], cudaEventDisableTiming));
    }
    CU(cudaEventCreateWithFlags(&e->ev_fork, cudaEventDisableTiming));
    CU(e->d_logmax.ensure(1));
    CU(e->d_nact.ensure(e->npairs()));
    CU(e->d_counters.ensure(MAX_CHUNKS));
    CU(e->d_qcounts.ensure(MAX_CHUNKS));
    *out = e.release();
    return JQC_OK;
}

extern "C" void jqc_engine_destroy(jqc_engine* e)
{
    if (!e) return;
    cudaSetDevice(e->device);
    for (auto ev : e->ev) cudaEventDestroy(ev);
    for (int i = 0; i < jqc_engine::NAUX; i++) {
        if (e->aux[i]) cudaStreamDestroy(e->aux[i]);
        if (e->ev_join[i]) cudaEventDestroy(e->ev_join[i]);
    }
    if (e->ev_fork) cudaEventDestroy(e->ev_fork);
    delete e;
}

extern "C" int jqc_engine_nao(const jqc_engine* e) { return e ? e->nao : -1; }
extern "C" int jqc_engine_mol_nao(const jqc_engine* e) { return e ? e->mol_nao : -1; }

extern "C" int jqc_engine_set_shard(jqc_engine* e, int rank, int world)
{
    if (!e || world < 1 || rank < 0 || rank >= world) return fail(JQC_EINVAL, "bad shard");
    e->rank = rank;
    e->world = world;
    return JQC_OK;
}

extern "C" int jqc_set_profiling(jqc_engine* e, int enabled)
{
    if (!e) return fail(JQC_EINVAL, "null engine");
    e->profiling = enabled != 0;
    return JQC_OK;
}

// ---------------------------------------------------------------------------------------
static int get_qdata(jqc_engine* e, double omega, QData** out)
{
    auto it = e->qcache.find(omega);
    if (it != e->qcache.end()) { *out = it->second.get(); return JQC_OK; }
    std::unique_ptr<QData> qd(new QData);
    const int nbas = e->nbas, nt = e->nt;
    CU(qd->q.ensure((size_t)nbas * nbas));
    {
        const int nfm = (e->lmax + 1) * (e->lmax + 2) / 2;
        const int blk = nfm * nfm * nfm * nfm;
        // scratch = one integral block per resident thread: bounded to ~1 GiB (g shells: 405 KB per thread)
        const int threads = 64;
        int blocks = std::max(1, std::min(e->nsm * 2, (nbas * (nbas + 1) / 2 + threads - 1) / threads));
        blocks = std::max(1, std::min(blocks, (int)((size_t(1) << 30) / ((size_t)threads * blk * sizeof(double)))));
        DevBuf<GenScratch> scratch;
        DevBuf<double> blocksbuf;
        CU(scratch.ensure((size_t)threads * blocks));
        CU(blocksbuf.ensure((size_t)threads * blocks * blk));
        q_cond_kernel<<<blocks, threads>>>(e->d_basis.p, e->d_angs.p, e->d_nprims.p, e->d_pad.p, nbas, e->mol_cart,
                                          e->xt, omega, scratch.p, blocksbuf.p, blk, qd->q.p);
        CU(cudaGetLastError());
        CU(cudaDeviceSynchronize());
    }
    DevBuf<float> tq;
    CU(tq.ensure((size_t)nt * nt));
    tile_max_kernel<<<(nt * nt + 255) / 256, 256>>>(qd->q.p, nbas, tq.p);
    CU(cudaGetLastError());
    std::vector<float> h_tq((size_t)nt * nt);
    CU(cudaMemcpy(h_tq.data(), tq.p, h_tq.size() * sizeof(float), cudaMemcpyDeviceToHost));
    // per group pair (gi >= gj): tiles sorted by q descending; tiles that can never pass any
    // realistic cutoff (q = -100 pads) are dropped
    std::vector<int> tiles;
    std::vector<float> tiles_q;
    qd->h_list_off.assign(1, 0);
    for (int gi = 0; gi < e->ngroups; gi++)
        for (int gj = 0; gj <= gi; gj++) {
            std::vector<std::pair<float, int>> v;
            for (int ti = e->goff[gi] / JQC_TILE; ti < e->goff[gi + 1] / JQC_TILE; ti++)
                for (int tj = e->goff[gj] / JQC_TILE; tj < e->goff[gj + 1] / JQC_TILE; tj++) {
                    if (gi == gj && tj > ti) continue;
                    const float qv = h_tq[(size_t)ti * nt + tj];
                    if (qv > -90.f) v.emplace_back(-qv, ti * nt + tj);
                }
            std::sort(v.begin(), v.end());
            for (auto& pr : v) { tiles.push_back(pr.second); tiles_q.push_back(-pr.first); }
            qd->h_list_off.push_back((int)tiles.size());
        }
    CU(qd->tiles.upload(tiles));
    CU(qd->tiles_q.upload(tiles_q));
    CU(qd->list_off.upload(qd->h_list_off));
    {   // pair lists for the brick kernel
        std::vector<float> hq((size_t)nbas * nbas);
        CU(cudaMemcpy(hq.data(), qd->q.p, hq.size() * sizeof(float), cudaMemcpyDeviceToHost));
        std::vector<ushort2> kl;
        std::vector<float> kl_q, kl_tq, j_q, j_tq;
        std::vector<unsigned short> j_idx;
        std::vector<ushort2> j_pairs;      // (a, b) in bra-list order, for the primitive-pair table
        std::vector<int> j_off;
        qd->h_pair_off.assign(1, 0);
        struct Ent { int bucket; float q; unsigned short a, b; };
        std::vector<Ent> v;
        for (int ga = 0; ga < e->ngroups; ga++)
            for (int gb = 0; gb <= ga; gb++) {
                v.clear();
                float qmax = -INFINITY;
                qd->h_joff_off.push_back((int)j_off.size());
                for (int a = e->goff[ga]; a < e->goff[ga + 1]; a++) {
                    j_off.push_back((int)j_idx.size());
                    const size_t row0 = v.size();
                    const int bend = ga == gb ? a + 1 : e->goff[gb + 1];
                    for (int b = e->goff[gb]; b < bend; b++) {
                        const float qv = hq[(size_t)a * nbas + b];
                        if (!(qv > -90.f)) continue;
                        v.push_back({(a - e->goff[ga]) / 32, qv, (unsigned short)a, (unsigned short)b});
                        qmax = std::max(qmax, qv);
                    }
                    // bra role: this row by q descending (ties by shell index: deterministic)
                    std::vector<Ent> row(v.begin() + row0, v.end());
                    std::sort(row.begin(), row.end(), [](const Ent& x, const Ent& y) { return x.q != y.q ? x.q > y.q : x.b < y.b; });
                    for (auto& r : row) {
                        j_idx.push_back(r.b);
                        j_pairs.push_back(make_ushort2(r.a, r.b));
                        j_q.push_back(r.q);
                        j_tq.push_back(h_tq[(size_t)(r.a / JQC_TILE) * nt + r.b / JQC_TILE]);
                    }
                }
                j_off.push_back((int)j_idx.size());
                std::sort(v.begin(), v.end(), [](const Ent& x, const Ent& y) {
                    if (x.bucket != y.bucket) return x.bucket < y.bucket;
                    if (x.q != y.q) return x.q > y.q;
                    return x.a != y.a ? x.a < y.a : x.b < y.b;
                });
                for (auto& r : v) {
                    kl.push_back(make_ushort2(r.a, r.b));
                    kl_q.push_back(r.q);
                    kl_tq.push_back(h_tq[(size_t)(r.a / JQC_TILE) * nt + r.b / JQC_TILE]);
                }
                qd->h_pair_off.push_back((int)kl.size());
                qd->h_qmax.push_back(qmax);
            }
        CU(qd->kl.upload(kl));
        CU(qd->kl_q.upload(kl_q));
        CU(qd->kl_tq.upload(kl_tq));
        CU(qd->j_idx.upload(j_idx));
        CU(qd->j_q.upload(j_q));
        CU(qd->j_tq.upload(j_tq));
        CU(qd->j_off.upload(j_off));
        // primitive-pair tables of both lists
        DevBuf<ushort2> d_jpairs;
        CU(d_jpairs.upload(j_pairs));
        size_t tot = 0;
        for (int ga = 0, P = 0; ga < e->ngroups; ga++)
            for (int gb = 0; gb <= ga; gb++, P++) {
                qd->h_tab_off.push_back(tot);
                tot += (size_t)(qd->h_pair_off[P + 1] - qd->h_pair_off[P]) * e->gnp[ga] * e->gnp[gb] * 8;
            }
        CU(qd->ket_tab.ensure(std::max<size_t>(tot, 1)));
        CU(qd->bra_tab.ensure(std::max<size_t>(tot, 1)));
        for (int ga = 0, P = 0; ga < e->ngroups; ga++)
            for (int gb = 0; gb <= ga; gb++, P++) {
                const int n = qd->h_pair_off[P + 1] - qd->h_pair_off[P];
                if (n == 0) continue;
                const long long work = (long long)n * e->gnp[ga] * e->gnp[gb];
                const unsigned blocks = (unsigned)((work + 255) / 256);
                pair_prim_kernel<<<blocks, 256>>>(e->d_basis.p, qd->kl.p + qd->h_pair_off[P], n, e->gnp[ga], e->gnp[gb],
                                                 qd->ket_tab.p + qd->h_tab_off[P]);
                pair_prim_kernel<<<blocks, 256>>>(e->d_basis.p, d_jpairs.p + qd->h_pair_off[P], n, e->gnp[ga], e->gnp[gb],
                                                 qd->bra_tab.p + qd->h_tab_off[P]);
            }
        CU(cudaGetLastError());
        CU(cudaDeviceSynchronize());
    }
    *out = qd.get();
    e->qcache[omega] = std::move(qd);
    return JQC_OK;
}

extern "C" int jqc_q_matrix(jqc_engine* e, double omega, const float** q_dev)
{
    if (!e || !q_dev) return fail(JQC_EINVAL, "null argument");
    if (omega < 0) return fail(JQC_EINVAL, "short ranged J/K not supported");
    CU(cudaSetDevice(e->device));
    QData* qd = nullptr;
    int rc = get_qdata(e, omega, &qd);
    if (rc) return rc;
    *q_dev = qd->q.p;
    return JQC_OK;
}

// ---------------------------------------------------------------------------------------
static int launch_from_mol(jqc_engine* e, const double* mol, int n, double* kern, bool transpose, cudaStream_t st)
{
    if (e->nao == 0 || n == 0) return JQC_OK;
    dim3 grid(e->nao, (e->nao + 127) / 128, n);   // rows on grid.x (no 65535 limit)
    dm_from_mol_kernel<<<grid, 128, 0, st>>>(mol, e->mol_nao, kern, e->nao, e->d_ao2shell.p, e->d_ao_loc.p,
                                            e->d_angs.p, e->d_mol_off.p, e->xt, transpose ? 1 : 0);
    CU(cudaGetLastError());
    return JQC_OK;
}

static int launch_to_mol(jqc_engine* e, const double* kern, int n, int n_half, int mode, double* mol, cudaStream_t st)
{
    if (e->mol_nao == 0 || n == 0) return JQC_OK;
    dim3 grid(e->mol_nao, (e->mol_nao + 127) / 128, n);
    dm_to_mol_kernel<<<grid, 128, 0, st>>>(kern, e->nao, n_half, mode, mol, e->mol_nao, e->d_molao_parent.p,
                                          e->d_molao_m.p, e->d_child_ptr.p, e->d_child_list.p, e->d_ao_loc.p,
                                          e->d_angs.p, e->xt);
    CU(cudaGetLastError());
    return JQC_OK;
}

extern "C" int jqc_dm_from_mol(jqc_engine* e, const double* mol_dev, int n, double* kern_dev, void* stream)
{
    if (!e || !mol_dev || !kern_dev || n < 0) return fail(JQC_EINVAL, "bad argument");
    CU(cudaSetDevice(e->device));
    return launch_from_mol(e, mol_dev, n, kern_dev, false, (cudaStream_t)stream);
}

extern "C" int jqc_dm_to_mol(jqc_engine* e, const double* kern_dev, int n, double* mol_dev, void* stream)
{
    if (!e || !mol_dev || !kern_dev || n < 0) return fail(JQC_EINVAL, "bad argument");
    CU(cudaSetDevice(e->device));
    return launch_to_mol(e, kern_dev, n, n, 0, mol_dev, (cudaStream_t)stream);
}

// ---------------------------------------------------------------------------------------
extern "C" int jqc_build_partial(jqc_engine* e, const double* dm_dev, int n_dm, int hermi, int with_j, int with_k,
                                 double omega, double cutoff_fp64, double cutoff_fp32, double** partial_dev,
                                 size_t* partial_len, void* stream)
{
    if (!e || !dm_dev) return fail(JQC_EINVAL, "null argument");
    if (n_dm < 1) return fail(JQC_EINVAL, "n_dm must be >= 1");
    if (!with_j && !with_k) return fail(JQC_EINVAL, "with_j or with_k required");
    if (omega < 0) return fail(JQC_EINVAL, "short ranged J/K not supported");
    if (!(cutoff_fp64 > 0) || !(cutoff_fp32 > 0)) return fail(JQC_EINVAL, "cutoffs must be positive");
    CU(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    QData* qd = nullptr;
    int rc = get_qdata(e, omega, &qd);
    if (rc) return rc;

    const int nao = e->nao, nbas = e->nbas;
    const size_t nao2 = (size_t)nao * nao;
    const int neff = hermi == 1 ? n_dm : 2 * n_dm;
    CU(e->d_dm.ensure(std::max<size_t>(neff * nao2, 1)));
    CU(e->d_vjk.ensure(std::max<size_t>(2 * neff * nao2, 1)));
    CU(e->d_cond.ensure((size_t)nbas * nbas));
    CU(e->d_logd.ensure((size_t)nbas * nbas));

    // 1. AO transform in (+ transposed copies when hermi != 1, jk.py:189-192)
    rc = launch_from_mol(e, dm_dev, n_dm, e->d_dm.p, false, st);
    if (rc) return rc;
    if (hermi != 1) {
        rc = launch_from_mol(e, dm_dev, n_dm, e->d_dm.p + n_dm * nao2, true, st);
        if (rc) return rc;
    }
    // Mixed precision (jk.py:93-96, 241-328): quartets whose estimate lies in (cutoff_fp32, cutoff_fp64]
    // go to the FP32 variant of the brick kernel, which reads a float copy of the density.
    const bool mixed = cutoff_fp64 > cutoff_fp32 && e->use_brick && neff == 1 && !e->small_tiles && e->use_fp32;
    if (mixed) {
        CU(e->d_dm32.ensure(std::max<size_t>(nao2, 1)));
        const unsigned blocks = (unsigned)std::min<size_t>((nao2 + 255) / 256, 65535u * 16);
        to_float_kernel<<<blocks, 256, 0, st>>>(e->d_dm.p, e->d_dm32.p, nao2);
        CU(cudaGetLastError());
    }
    // 2. density pooling on the first n_dm matrices, log, global max
    dm_pool_kernel<<<nbas, 256, nbas * sizeof(float), st>>>(e->d_dm.p, n_dm, nao, nbas, e->d_ao_loc.p, e->d_ao2shell.p,
                                                          e->d_cond.p);
    CU(cudaGetLastError());
    {
        const int neg_inf_ordered = (int)0xFF800000 ^ 0x7FFFFFFF;   // float_to_ordered(-inf)
        CU(cudaMemcpyAsync(e->d_logmax.p, &neg_inf_ordered, sizeof(int), cudaMemcpyHostToDevice, st));
        dim3 grid(nbas, (nbas + 127) / 128);
        dm_log_kernel<<<grid, 128, 0, st>>>(e->d_cond.p, nbas, hermi == 1 ? 1 : 0, e->d_logd.p, e->d_logmax.p);
        CU(cudaGetLastError());
    }
    // 3. active tile counts per group pair
    const int npairs = e->npairs();
    active_tiles_kernel<<<(npairs + 127) / 128, 128, 0, st>>>(qd->tiles_q.p, qd->list_off.p, npairs, e->d_logmax.p,
                                                             e->d_nact.p);
    CU(cudaGetLastError());
    CU(cudaMemsetAsync(e->d_vjk.p, 0, 2 * neff * nao2 * sizeof(double), st));
    CU(cudaMemsetAsync(e->d_counters.p, 0, MAX_CHUNKS * sizeof(unsigned), st));
    CU(cudaMemsetAsync(e->d_qcounts.p, 0, MAX_CHUNKS * sizeof(unsigned long long), st));
    // The only host round trip of a build: the per-group-pair active tile counts (a few hundred
    // ints) so that no empty chunk is ever launched.  It happens before any heavy kernel is
    // enqueued, i.e. with an empty pipeline (the reference syncs here too, jk.py:183).
    std::vector<int> nact(npairs);
    CU(cudaMemcpyAsync(nact.data(), e->d_nact.p, npairs * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));

    // 4. group-quartet loop (order of jk.py:145-151, 209: reversed, heavy classes first)
    double* vj = e->d_vjk.p;
    double* vk = e->d_vjk.p + neff * nao2;
    const float log_cut = (float)std::log(std::min(cutoff_fp32, cutoff_fp64));
    const float log_cut64 = (float)std::log(cutoff_fp64);
    const int variant = (with_j ? 1 : 0) | (with_k ? 2 : 0);
    e->chunks.clear();
    e->launches = 0;
    size_t nev = 0;
    bool queue_ready = false;
    const bool fork = e->use_aux && !e->profiling;
    int n_brick = 0;
    if (fork) {
        CU(cudaEventRecord(e->ev_fork, st));
        for (int i = 0; i < jqc_engine::NAUX; i++) CU(cudaStreamWaitEvent(e->aux[i], e->ev_fork, 0));
    }
    for (int gi = e->ngroups - 1; gi >= 0; gi--)
    for (int gj = gi; gj >= 0; gj--)
    for (int gk = gi; gk >= 0; gk--)
    for (int gl = gk; gl >= 0; gl--) {
        const int pij = jqc_engine::pair_id(gi, gj), pkl = jqc_engine::pair_id(gk, gl);
        const int n_ij_all = nact[pij];
        const int n_kl = nact[pkl];
        if (n_ij_all == 0 || n_kl == 0) continue;
        const int li = e->gl[gi], lj = e->gl[gj], lk = e->gl[gk], ll = e->gl[gl];
        const int key = ((li * 5 + lj) * 5 + lk) * 5 + ll;
        const long long pw = (long long)e->gnp[gi] * e->gnp[gj] * e->gnp[gk] * e->gnp[gl];
        const bool brick_small = brick_shape(li, lj, lk, ll).fits;
        const bool on_brick = e->use_brick && neff == 1 && !e->small_tiles &&
                              (brick_small || (e->use_bwarp && jk_bwarp_supported(li, lj, lk, ll, e->use_bwarp)));
        // FP32 kernel of this class for the mixed-precision band: brick variant up to JQC_SMALL_N
        // integrals, brick-scheduled multi-lane variant above (up to f shells)
        const bool f32_brick = brick_shape(li, lj, lk, ll, true).fits;
        const int band_variant = f32_brick ? 16 : (jk_bwarp_supported(li, lj, lk, ll, 2) ? 24 : 0);
        const bool band = mixed && band_variant != 0;
        const int n_kl_pairs = qd->h_pair_off[pkl + 1] - qd->h_pair_off[pkl];
        const int n_ij_pairs = qd->h_pair_off[pij + 1] - qd->h_pair_off[pij];
        BrickArgs b;
        if (on_brick || band) {
            if (n_kl_pairs == 0 || n_ij_pairs == 0) continue;
            b.nao = nao; b.nbas = nbas;
            b.npi = e->gnp[gi]; b.npj = e->gnp[gj]; b.npk = e->gnp[gk]; b.npl = e->gnp[gl];
            b.basis = e->d_basis.p; b.dm = e->d_dm.p; b.vj = vj; b.vk = vk; b.omega = omega;
            b.logd = e->d_logd.p; b.log_max_ordered = e->d_logmax.p;
            b.cutoff = band ? std::max(log_cut, log_cut64) : log_cut;
            b.cutoff_hi = INFINITY;
            b.dm32 = nullptr;
            b.kl = qd->kl.p + qd->h_pair_off[pkl];
            b.kl_q = qd->kl_q.p + qd->h_pair_off[pkl];
            b.kl_tq = qd->kl_tq.p + qd->h_pair_off[pkl];
            b.n_kl = n_kl_pairs;
            b.i_first = e->goff[gi];
            b.i_count = e->goff[gi + 1] - e->goff[gi];
            b.j_off = qd->j_off.p + qd->h_joff_off[pij];
            b.j_idx = qd->j_idx.p; b.j_q = qd->j_q.p; b.j_tq = qd->j_tq.p;
            b.j_base = qd->h_pair_off[pij];
            b.bra_tab = qd->bra_tab.p + qd->h_tab_off[pij];
            b.ket_tab = qd->ket_tab.p + qd->h_tab_off[pkl];
            b.qmax_ij = qd->h_qmax[pij];
            b.tri = gi == gk;
            b.n_ij = n_ij_pairs;
            b.ichunk_req = e->brick_ichunk;
            b.n_blk = b.ichunk = b.n_ichunk = b.jsplit = 0;      // set by the launcher (brick_decompose)
            b.rank = e->rank; b.world = e->world;
        }
        // one launch of the brick family (FP64 share, or the FP32 band) with its own task counter
        auto brick_family_launch = [&](int var, bool fp32) -> int {
            if ((int)e->chunks.size() >= MAX_CHUNKS) return fail(JQC_ENOMEM, "too many task chunks");
            const int cid = (int)e->chunks.size();
            b.work = e->d_counters.p + cid;
            b.qcount = e->d_qcounts.p + cid;
            cudaEvent_t e0 = nullptr, e1 = nullptr;
            if (e->profiling) {
                while (e->ev.size() < nev + 2) { cudaEvent_t x; CU(cudaEventCreate(&x)); e->ev.push_back(x); }
                e0 = e->ev[nev++]; e1 = e->ev[nev++];
                CU(cudaEventRecord(e0, st));
            }
            CU(jk_brick_launch(li, lj, lk, ll, var, b, e->nsm, fork ? e->aux[n_brick++ % jqc_engine::NAUX] : st));
            if (e->profiling) CU(cudaEventRecord(e1, st));
            e->launches += 1;
            e->chunks.push_back({key, pw, fp32});
            return JQC_OK;
        };
        if (band) {
            // quartets with cutoff_fp32 < estimate <= cutoff_fp64 (screen_jk_tasks.cu:258-261)
            const float lo = b.cutoff;
            b.cutoff = log_cut;
            b.cutoff_hi = log_cut64;
            b.dm32 = e->d_dm32.p;
            rc = brick_family_launch(variant | band_variant, true);
            if (rc) return rc;
            b.cutoff = lo;
            b.cutoff_hi = INFINITY;
            b.dm32 = nullptr;
        }
        if (on_brick) {
            rc = brick_family_launch(variant | (brick_small ? 0 : 8), false);
            if (rc) return rc;
            continue;
        }
        // quartet-list path: this rank owns entries shard_entry(0, rank, world), shard_entry(1, ...), ... of the
        // q-sorted ij tile list (slots past the end of the list are masked in the kernel)
        const int n_ij = (n_ij_all + e->world - 1) / e->world;
        if (n_ij <= 0) continue;
        // chunk so that 256 * ij_tiles * kl_tiles <= queue capacity (and the grid's y extent <= 65535)
        const int kl_chunk = std::min({n_kl, e->kl_chunk_max, (int)(e->queue_cap / 256)});
        const int ij_chunk = std::max(1, (int)std::min<size_t>({(size_t)n_ij, e->queue_cap / 256 / kl_chunk, (size_t)32767}));
        if (!queue_ready) {   // sized once per build from the longest active tile list
            const size_t mx = (size_t)*std::max_element(nact.begin(), nact.end());
            CU(e->d_queue.ensure(std::max<size_t>(256, std::min(e->queue_cap, 256 * mx * std::min<size_t>(mx, e->kl_chunk_max)))));
            queue_ready = true;
        }
        for (int ij0 = 0; ij0 < n_ij; ij0 += ij_chunk)
        for (int kl0 = 0; kl0 < n_kl; kl0 += kl_chunk) {
            if ((int)e->chunks.size() >= MAX_CHUNKS) return fail(JQC_ENOMEM, "too many task chunks");
            const int cid = (int)e->chunks.size();
            ScreenArgs s;
            s.nbas = nbas;
            s.q = qd->q.p;
            s.logd = e->d_logd.p;
            s.log_max_ordered = e->d_logmax.p;
            s.tiles_ij = qd->tiles.p + qd->h_list_off[pij];
            s.tiles_kl = qd->tiles.p + qd->h_list_off[pkl];
            s.tileq_kl = qd->tiles_q.p + qd->h_list_off[pkl];
            s.nact_ij = e->d_nact.p + pij;
            s.nact_kl = e->d_nact.p + pkl;
            s.ij_begin = ij0;
            s.ij_count = std::min(ij_chunk, n_ij - ij0);
            s.kl_begin = kl0;
            s.kl_count = std::min(kl_chunk, n_kl - kl0);
            s.rank = e->rank;
            s.world = e->world;
            s.cutoff = band ? std::max(log_cut, log_cut64) : log_cut;
            s.do_j = with_j;
            s.do_k = with_k;
            s.queue = e->d_queue.p;
            s.counter = e->d_counters.p + cid;
            s.qcount = e->d_qcounts.p + cid;
            s.tile_mode = (e->small_tiles && jk_uses_tiles(li, lj, lk, ll)) ? 1 : 0;
            cudaEvent_t e0 = nullptr, e1 = nullptr;
            if (e->profiling) {
                while (e->ev.size() < nev + 2) { cudaEvent_t x; CU(cudaEventCreate(&x)); e->ev.push_back(x); }
                e0 = e->ev[nev++]; e1 = e->ev[nev++];
                CU(cudaEventRecord(e0, st));
            }
            dim3 sgrid((s.kl_count + 31) / 32, (s.ij_count * 16 + 7) / 8);
            screen_tasks_kernel<false><<<sgrid, dim3(32, 8), 0, st>>>(s);
            CU(cudaGetLastError());
            JKArgs a;
            a.nao = nao;
            a.n_dm = neff;
            a.npi = e->gnp[gi]; a.npj = e->gnp[gj]; a.npk = e->gnp[gk]; a.npl = e->gnp[gl];
            a.basis = e->d_basis.p;
            a.dm = e->d_dm.p;
            a.vj = vj;
            a.vk = vk;
            a.omega = omega;
            a.quartets = e->d_queue.p;
            a.ntasks = e->d_counters.p + cid;
            CU(jk_launch(li, lj, lk, ll, variant | (s.tile_mode ? 4 : 0), a, e->nsm, st));
            if (e->profiling) CU(cudaEventRecord(e1, st));
            e->launches += 2;
            e->chunks.push_back({key, pw});
        }
    }
    if (fork) {
        for (int i = 0; i < jqc_engine::NAUX; i++) {
            CU(cudaEventRecord(e->ev_join[i], e->aux[i]));
            CU(cudaStreamWaitEvent(st, e->ev_join[i], 0));
        }
    }
    e->last_n = n_dm; e->last_neff = neff; e->last_hermi = hermi; e->last_j = with_j; e->last_k = with_k;
    e->built = true;
    if (partial_dev) *partial_dev = e->d_vjk.p;
    if (partial_len) *partial_len = 2 * neff * nao2;
    return JQC_OK;
}

// ---------------------------------------------------------------------------------------
// Nuclear gradient of the J/K energy (include/joltqc_b200.h), shared by both entry points:
//   nspin = 1: E_jk = (j_factor/2) tr(D J[D]) - (k_factor/4) tr(D K[D]) for one density D;
//   nspin = 2: E_U = (j_factor/2) tr(Dt J[Dt]) - (k_factor/2) sum_s tr(Ds K[Ds]) for the spin densities
//              Da, Db (dm_dev holds both) and Dt = Da + Db.
// Same front end as a J/K build (transform in, pooling, active tile lists, chunked group-quartet loop
// with the device queue), on the quartet-list path only.  The density scratch, the pooled density and the
// queue are shared with the J/K builds (stream-ordered); the [J || K] buffer, the chunk records and the
// task counters that jqc_finalize and jqc_last_stats read are not touched.
static int jk_energy_grad(jqc_engine* e, const double* dm_dev, int nspin, double j_factor, double k_factor,
                          double omega, double cutoff, const int* shell_atom, int natm, double* grad_dev,
                          long long* quartets, void* stream)
{
    if (!e || !dm_dev || !shell_atom || !grad_dev) return fail(JQC_EINVAL, "null argument");
    if (omega < 0) return fail(JQC_EINVAL, "short ranged J/K not supported");
    if (j_factor == 0.0 && k_factor == 0.0) return fail(JQC_EINVAL, "j_factor or k_factor must be non-zero");
    if (!(cutoff > 0)) return fail(JQC_EINVAL, "cutoff must be positive");
    if (natm < 1) return fail(JQC_EINVAL, "natm must be >= 1");
    for (int s = 0; s < e->nbas; s++)
        if (shell_atom[s] < -1 || shell_atom[s] >= natm) return fail(JQC_EINVAL, "shell_atom entry outside [-1, natm)");
    CU(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    QData* qd = nullptr;
    int rc = get_qdata(e, omega, &qd);
    if (rc) return rc;

    const int nao = e->nao, nbas = e->nbas, npairs = e->npairs();
    const size_t nao2 = (size_t)nao * nao;
    // kernel-side densities: D, or [Da | Db | Dt]
    CU(e->d_dm.ensure(std::max<size_t>((nspin == 1 ? 1 : 3) * nao2, 1)));
    CU(e->d_cond.ensure((size_t)nbas * nbas));
    CU(e->d_logd.ensure((size_t)nbas * nbas));
    if (nspin == 2) CU(e->d_glogdj.ensure((size_t)nbas * nbas));
    CU(e->d_gcounters.ensure(MAX_CHUNKS));
    CU(e->d_gqcounts.ensure(MAX_CHUNKS));
    CU(e->d_gshell.ensure((size_t)nbas * 3));
    CU(e->d_gatom.ensure(nbas));
    CU(cudaMemcpyAsync(e->d_gatom.p, shell_atom, nbas * sizeof(int), cudaMemcpyHostToDevice, st));

    // 1. AO transform in (and Dt = Da + Db), 2. pooling (hermi = 1), log, global max: d pools max_s |Ds|
    // (the K terms), dJ pools Dt (the J term); both logs raise the one global maximum.  3. active tile
    // counts (quadratic in D).
    rc = launch_from_mol(e, dm_dev, nspin, e->d_dm.p, false, st);
    if (rc) return rc;
    if (nspin == 2) {
        const unsigned blocks = (unsigned)std::min<size_t>((nao2 + 255) / 256, 65535u * 16);
        dm_spin_sum_kernel<<<blocks, 256, 0, st>>>(e->d_dm.p, e->d_dm.p + nao2, e->d_dm.p + 2 * nao2, nao2);
        CU(cudaGetLastError());
    }
    {
        const int neg_inf_ordered = (int)0xFF800000 ^ 0x7FFFFFFF;   // float_to_ordered(-inf)
        CU(cudaMemcpyAsync(e->d_logmax.p, &neg_inf_ordered, sizeof(int), cudaMemcpyHostToDevice, st));
        dim3 grid(nbas, (nbas + 127) / 128);
        dm_pool_kernel<<<nbas, 256, nbas * sizeof(float), st>>>(e->d_dm.p, nspin, nao, nbas, e->d_ao_loc.p,
                                                              e->d_ao2shell.p, e->d_cond.p);
        CU(cudaGetLastError());
        dm_log_kernel<<<grid, 128, 0, st>>>(e->d_cond.p, nbas, 1, e->d_logd.p, e->d_logmax.p);
        CU(cudaGetLastError());
        if (nspin == 2) {
            dm_pool_kernel<<<nbas, 256, nbas * sizeof(float), st>>>(e->d_dm.p + 2 * nao2, 1, nao, nbas, e->d_ao_loc.p,
                                                                  e->d_ao2shell.p, e->d_cond.p);
            CU(cudaGetLastError());
            dm_log_kernel<<<grid, 128, 0, st>>>(e->d_cond.p, nbas, 1, e->d_glogdj.p, e->d_logmax.p);
            CU(cudaGetLastError());
        }
    }
    active_tiles_grad_kernel<<<(npairs + 127) / 128, 128, 0, st>>>(qd->tiles_q.p, qd->list_off.p, npairs, e->d_logmax.p,
                                                                  e->d_nact.p);
    CU(cudaGetLastError());
    CU(cudaMemsetAsync(e->d_gshell.p, 0, (size_t)nbas * 3 * sizeof(double), st));
    CU(cudaMemsetAsync(e->d_gcounters.p, 0, MAX_CHUNKS * sizeof(unsigned), st));
    CU(cudaMemsetAsync(e->d_gqcounts.p, 0, MAX_CHUNKS * sizeof(unsigned long long), st));
    std::vector<int> nact(npairs);
    CU(cudaMemcpyAsync(nact.data(), e->d_nact.p, npairs * sizeof(int), cudaMemcpyDeviceToHost, st));
    CU(cudaStreamSynchronize(st));

    // 4. group-quartet loop of the quartet-list path (jqc_build_partial), heavy classes first
    const float log_cut = (float)std::log(cutoff);
    int nchunks = 0;
    bool queue_ready = false;
    for (int gi = e->ngroups - 1; gi >= 0; gi--)
    for (int gj = gi; gj >= 0; gj--)
    for (int gk = gi; gk >= 0; gk--)
    for (int gl = gk; gl >= 0; gl--) {
        const int pij = jqc_engine::pair_id(gi, gj), pkl = jqc_engine::pair_id(gk, gl);
        const int n_ij_all = nact[pij];
        const int n_kl = nact[pkl];
        if (n_ij_all == 0 || n_kl == 0) continue;
        const int li = e->gl[gi], lj = e->gl[gj], lk = e->gl[gk], ll = e->gl[gl];
        const int n_ij = (n_ij_all + e->world - 1) / e->world;
        if (n_ij <= 0) continue;
        const int kl_chunk = std::min({n_kl, e->kl_chunk_max, (int)(e->queue_cap / 256)});
        const int ij_chunk = std::max(1, (int)std::min<size_t>({(size_t)n_ij, e->queue_cap / 256 / kl_chunk, (size_t)32767}));
        if (!queue_ready) {
            const size_t mx = (size_t)*std::max_element(nact.begin(), nact.end());
            CU(e->d_queue.ensure(std::max<size_t>(256, std::min(e->queue_cap, 256 * mx * std::min<size_t>(mx, e->kl_chunk_max)))));
            queue_ready = true;
        }
        for (int ij0 = 0; ij0 < n_ij; ij0 += ij_chunk)
        for (int kl0 = 0; kl0 < n_kl; kl0 += kl_chunk) {
            if (nchunks >= MAX_CHUNKS) return fail(JQC_ENOMEM, "too many task chunks");
            const int cid = nchunks++;
            ScreenArgs s;
            s.nbas = nbas;
            s.q = qd->q.p;
            s.logd = e->d_logd.p;
            s.logd_j = nspin == 1 ? e->d_logd.p : e->d_glogdj.p;
            s.log_max_ordered = e->d_logmax.p;
            s.tiles_ij = qd->tiles.p + qd->h_list_off[pij];
            s.tiles_kl = qd->tiles.p + qd->h_list_off[pkl];
            s.tileq_kl = qd->tiles_q.p + qd->h_list_off[pkl];
            s.nact_ij = e->d_nact.p + pij;
            s.nact_kl = e->d_nact.p + pkl;
            s.ij_begin = ij0;
            s.ij_count = std::min(ij_chunk, n_ij - ij0);
            s.kl_begin = kl0;
            s.kl_count = std::min(kl_chunk, n_kl - kl0);
            s.rank = e->rank;
            s.world = e->world;
            s.cutoff = log_cut;
            s.do_j = j_factor != 0.0;
            s.do_k = k_factor != 0.0;
            s.queue = e->d_queue.p;
            s.counter = e->d_gcounters.p + cid;
            s.qcount = e->d_gqcounts.p + cid;
            s.tile_mode = 0;
            dim3 sgrid((s.kl_count + 31) / 32, (s.ij_count * 16 + 7) / 8);
            screen_tasks_kernel<true><<<sgrid, dim3(32, 8), 0, st>>>(s);
            CU(cudaGetLastError());
            GradArgs a;
            a.nao = nao;
            a.npi = e->gnp[gi]; a.npj = e->gnp[gj]; a.npk = e->gnp[gk]; a.npl = e->gnp[gl];
            a.basis = e->d_basis.p;
            a.dm = e->d_dm.p;
            a.dm_b = nspin == 1 ? nullptr : e->d_dm.p + nao2;
            a.dm_t = nspin == 1 ? nullptr : e->d_dm.p + 2 * nao2;
            a.j_factor4 = 4.0 * j_factor;
            a.k_factor = nspin == 1 ? k_factor : 2.0 * k_factor;
            a.omega = omega;
            a.quartets = e->d_queue.p;
            a.ntasks = e->d_gcounters.p + cid;
            a.gshell = e->d_gshell.p;
            CU(jk_grad_launch(li, lj, lk, ll, nspin, a, e->nsm, st));
        }
    }
    // 5. shells -> atoms
    grad_shell_to_atom_kernel<<<(3 * natm + 127) / 128, 128, 0, st>>>(e->d_gshell.p, e->d_gatom.p, nbas, natm, grad_dev);
    CU(cudaGetLastError());
    if (quartets) {
        std::vector<unsigned long long> h(std::max(nchunks, 1), 0ull);
        if (nchunks) CU(cudaMemcpyAsync(h.data(), e->d_gqcounts.p, nchunks * sizeof(unsigned long long), cudaMemcpyDeviceToHost, st));
        CU(cudaStreamSynchronize(st));
        long long n = 0;
        for (int c = 0; c < nchunks; c++) n += (long long)h[c];
        *quartets = n;
    }
    return JQC_OK;
}

extern "C" int jqc_jk_energy_grad(jqc_engine* e, const double* dm_dev, double j_factor, double k_factor, double omega,
                                  double cutoff, const int* shell_atom, int natm, double* grad_dev, long long* quartets,
                                  void* stream)
{
    return jk_energy_grad(e, dm_dev, 1, j_factor, k_factor, omega, cutoff, shell_atom, natm, grad_dev, quartets, stream);
}

extern "C" int jqc_jk_energy_grad_uhf(jqc_engine* e, const double* dm_dev, double j_factor, double k_factor,
                                      double omega, double cutoff, const int* shell_atom, int natm, double* grad_dev,
                                      long long* quartets, void* stream)
{
    return jk_energy_grad(e, dm_dev, 2, j_factor, k_factor, omega, cutoff, shell_atom, natm, grad_dev, quartets, stream);
}

extern "C" int jqc_finalize(jqc_engine* e, double* vj_dev, double* vk_dev, void* stream)
{
    if (!e) return fail(JQC_EINVAL, "null engine");
    if (!e->built) return fail(JQC_ESTATE, "jqc_finalize without jqc_build_partial");
    CU(cudaSetDevice(e->device));
    cudaStream_t st = (cudaStream_t)stream;
    const size_t nao2 = (size_t)e->nao * e->nao;
    const int n = e->last_n;
    if (e->last_j) {
        if (!vj_dev) return fail(JQC_EINVAL, "vj_dev is NULL but J was built");
        int rc = launch_to_mol(e, e->d_vjk.p, n, n, e->last_hermi == 1 ? 1 : 3, vj_dev, st);
        if (rc) return rc;
    }
    if (e->last_k) {
        if (!vk_dev) return fail(JQC_EINVAL, "vk_dev is NULL but K was built");
        int rc = launch_to_mol(e, e->d_vjk.p + e->last_neff * nao2, n, n, e->last_hermi == 1 ? 2 : 4, vk_dev, st);
        if (rc) return rc;
    }
    e->launches += (e->last_j ? 1 : 0) + (e->last_k ? 1 : 0);
    return JQC_OK;
}

extern "C" int jqc_get_jk(jqc_engine* e, const double* dm_dev, int n_dm, int hermi, int with_j, int with_k,
                          double omega, double cutoff_fp64, double cutoff_fp32, double* vj_dev, double* vk_dev,
                          void* stream)
{
    if (with_j && !vj_dev) return fail(JQC_EINVAL, "with_j needs vj_dev");
    if (with_k && !vk_dev) return fail(JQC_EINVAL, "with_k needs vk_dev");
    int rc = jqc_build_partial(e, dm_dev, n_dm, hermi, with_j, with_k, omega, cutoff_fp64, cutoff_fp32, nullptr,
                               nullptr, stream);
    if (rc) return rc;
    return jqc_finalize(e, vj_dev, vk_dev, stream);
}

extern "C" int jqc_get_jk_host(jqc_engine* e, const double* dm_host, int n_dm, int hermi, int with_j, int with_k,
                               double omega, double cutoff_fp64, double cutoff_fp32, double* vj_host, double* vk_host)
{
    if (!e || !dm_host) return fail(JQC_EINVAL, "null argument");
    if (n_dm < 1) return fail(JQC_EINVAL, "n_dm must be >= 1");
    if (with_j && !vj_host) return fail(JQC_EINVAL, "with_j needs vj_host");
    if (with_k && !vk_host) return fail(JQC_EINVAL, "with_k needs vk_host");
    CU(cudaSetDevice(e->device));
    const size_t sz = (size_t)n_dm * e->mol_nao * e->mol_nao;
    CU(e->d_stage_in.ensure(std::max<size_t>(sz, 1)));
    if (with_j) CU(e->d_stage_j.ensure(std::max<size_t>(sz, 1)));
    if (with_k) CU(e->d_stage_k.ensure(std::max<size_t>(sz, 1)));
    CU(cudaMemcpyAsync(e->d_stage_in.p, dm_host, sz * sizeof(double), cudaMemcpyHostToDevice, 0));
    int rc = jqc_get_jk(e, e->d_stage_in.p, n_dm, hermi, with_j, with_k, omega, cutoff_fp64, cutoff_fp32,
                        with_j ? e->d_stage_j.p : nullptr, with_k ? e->d_stage_k.p : nullptr, nullptr);
    if (rc) return rc;
    if (with_j) CU(cudaMemcpyAsync(vj_host, e->d_stage_j.p, sz * sizeof(double), cudaMemcpyDeviceToHost, 0));
    if (with_k) CU(cudaMemcpyAsync(vk_host, e->d_stage_k.p, sz * sizeof(double), cudaMemcpyDeviceToHost, 0));
    CU(cudaStreamSynchronize(0));
    return JQC_OK;
}

extern "C" int jqc_last_stats(jqc_engine* e, long long* counts, long long* prim_weighted, int* launches)
{
    if (!e) return fail(JQC_EINVAL, "null engine");
    if (!e->built) return fail(JQC_ESTATE, "no build yet");
    CU(cudaSetDevice(e->device));
    CU(cudaDeviceSynchronize());
    std::vector<unsigned long long> h(e->chunks.size());
    if (!h.empty()) CU(cudaMemcpy(h.data(), e->d_qcounts.p, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    if (counts) std::memset(counts, 0, 625 * sizeof(long long));
    if (prim_weighted) std::memset(prim_weighted, 0, 625 * sizeof(long long));
    std::fill(e->class_ms.begin(), e->class_ms.end(), 0.f);
    e->band_n[0] = e->band_n[1] = 0;
    e->band_ms[0] = e->band_ms[1] = 0.f;
    for (size_t c = 0; c < h.size(); c++) {
        e->band_n[e->chunks[c].fp32 ? 1 : 0] += (long long)h[c];
        if (counts) counts[e->chunks[c].key] += h[c];
        if (prim_weighted) prim_weighted[e->chunks[c].key] += (long long)h[c] * e->chunks[c].pw;
        if (e->profiling && e->ev.size() >= 2 * (c + 1)) {
            float ms = 0.f;
            if (cudaEventElapsedTime(&ms, e->ev[2 * c], e->ev[2 * c + 1]) == cudaSuccess) {
                e->class_ms[e->chunks[c].key] += ms;
                e->band_ms[e->chunks[c].fp32 ? 1 : 0] += ms;
            }
        }
    }
    if (launches) *launches = e->launches;
    return JQC_OK;
}

extern "C" int jqc_last_band_stats(jqc_engine* e, long long* quartets, float* ms)
{
    if (!e || !quartets) return fail(JQC_EINVAL, "null argument");
    int rc = jqc_last_stats(e, nullptr, nullptr, nullptr);
    if (rc) return rc;
    quartets[0] = e->band_n[0];
    quartets[1] = e->band_n[1];
    if (ms) { ms[0] = e->band_ms[0]; ms[1] = e->band_ms[1]; }
    return JQC_OK;
}

extern "C" int jqc_last_class_ms(jqc_engine* e, float* ms)
{
    if (!e || !ms) return fail(JQC_EINVAL, "null argument");
    if (!e->profiling) return fail(JQC_ESTATE, "profiling is off");
    int rc = jqc_last_stats(e, nullptr, nullptr, nullptr);
    if (rc) return rc;
    std::memcpy(ms, e->class_ms.data(), 625 * sizeof(float));
    return JQC_OK;
}

extern "C" int jqc_fp64_peak_probe(int device, double* tflops, double* sm_clock_mhz)
{
    if (!tflops) return fail(JQC_EINVAL, "null argument");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    double* out = nullptr;
    CU(cudaMalloc(&out, sizeof(double)));
    const int iters = 4096, threads = 256, blocks = prop.multiProcessorCount * 8;
    cudaEvent_t a, b;
    CU(cudaEventCreate(&a));
    CU(cudaEventCreate(&b));
    double best = 0.0;
    for (int rep = 0; rep < 5; rep++) {
        CU(cudaEventRecord(a));
        fp64_probe_kernel<<<blocks, threads>>>(out, iters, 1.0000001, 1e-9);
        CU(cudaEventRecord(b));
        CU(cudaEventSynchronize(b));
        float ms = 0;
        CU(cudaEventElapsedTime(&ms, a, b));
        const double flops = 2.0 * 64.0 * iters * (double)threads * blocks;
        if (rep > 0) best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    cudaEventDestroy(a);
    cudaEventDestroy(b);
    cudaFree(out);
    *tflops = best;
    if (sm_clock_mhz) {
        int khz = 0;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, device);
        *sm_clock_mhz = khz / 1000.0;
    }
    return JQC_OK;
}
