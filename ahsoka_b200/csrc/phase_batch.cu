// phase_batch.cu — host side of the C ABI (include/ahsoka_b200.h): uploads the CSR batch, runs the
// sm_100a kernels of k_project / k_score / k_cluster / k_thread on one stream, downloads the
// result.  No torch, no CPU fallback: without a usable CUDA device every entry point fails.
#include <algorithm>
#include <chrono>
#include <condition_variable>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <mutex>
#include <numeric>
#include <stdexcept>
#include <string>
#include <thread>
#include <vector>

#include "common.cuh"
#include "device_batch.cuh"
#include "k_project.cuh"
#include "k_front.cuh"
#include "k_score.cuh"
#include "k_chain.cuh"
#include "k_cluster_sparse.cuh"
#include "host_plan.hpp"
#include "k_thread.cuh"
#include "k_thread_canon.cuh"

namespace ahs {

static thread_local char g_err[512] = "";

static void set_err(const char* fmt, ...) { va_list ap; va_start(ap, fmt); vsnprintf(g_err, sizeof g_err, fmt, ap); va_end(ap); }

struct CudaFail { cudaError_t e; const char* what; int line; };
#define CK(call) do { cudaError_t _e = (call); if (_e != cudaSuccess) throw CudaFail{_e, #call, __LINE__}; } while (0)
struct LimitFail { std::string msg; };
struct ArgFail { std::string msg; };
struct PassThrough { int rc; std::string msg; };      // failure of one device thread of a multi-device call, re-raised by the caller

constexpr int MAX_READS_CLUSTER = 65535;       // 16-bit node ids in the edge keys of k_cluster_sparse (chains above CC_MAXN reads)
constexpr int MAX_POSITIONS = 32767;
constexpr int64_t MAX_READS_CHAIN = (int64_t)1 << 20;        // distinct read names per chain (k_read_rank is quadratic in them)
constexpr int64_t MAX_BIG_W_BYTES = (int64_t)48 << 30;       // dense weight matrices of the chains above CC_MAXN reads, per call and device

// ------------------------------------------------------------------ memory pools (persist per device)
struct Pool {
    struct Chunk { char* p; size_t cap, used; };
    std::vector<Chunk> chunks; bool host;
    explicit Pool(bool h) : host(h) {}
    void reset() { for (auto& c : chunks) c.used = 0; }
    void* alloc(size_t bytes) {
        bytes = (bytes + 255) & ~(size_t)255;
        if (bytes == 0) bytes = 256;
        for (auto& c : chunks) if (c.cap - c.used >= bytes) { void* r = c.p + c.used; c.used += bytes; return r; }
        size_t cap = std::max(bytes, (size_t)(host ? 64 : 256) << 20);
        Chunk c; c.cap = cap; c.used = bytes;
        if (host) CK(cudaHostAlloc((void**)&c.p, cap, cudaHostAllocPortable)); else CK(cudaMalloc((void**)&c.p, cap));
        chunks.push_back(c);
        return c.p;
    }
    template <class T> T* get(size_t n) { return (T*)alloc(n * sizeof(T)); }
    void release() { for (auto& c : chunks) { if (host) cudaFreeHost(c.p); else cudaFree(c.p); } chunks.clear(); }
};

// streams and events of one pipeline in flight (a call phases its chains in up to N_LANES chunks, chunk k+1 uploading
// and projecting while chunk k clusters).  ev[0..6]: stage boundaries of a pass (collect_times); ev[7], ev[8] of lane 0:
// the call's own events (DeviceJob)
struct Lane {
    cudaStream_t stream = nullptr, stream2 = nullptr;
    cudaEvent_t ev[9], ev_cells = nullptr, ev_en[8], ev_fork = nullptr, ev_join[8], ev_up = nullptr;
};
constexpr int N_LANES = 4;

struct Ctx {
    int device = -1; Lane lanes[N_LANES]; cudaStream_t side[8]; Pool dev{false}, pin{true}, outp{true};
    int64_t *d_ln = nullptr, *d_ln1 = nullptr; int sms = 148; bool out_busy = false;
    CanonTables canon{};                                     // neighbour tables of k_thread_canon (ploidy 5, 6)
    size_t smem_optin = 0;
    std::mutex mu;
};
static std::mutex g_ctx_mu;
static Ctx* g_ctx[64] = {nullptr};

// ------------------------------------------------------------------ shared-memory scoring + cluster editing: size classes
// Cluster editing: a class = (largest n, threads per block, pair slots per thread).  The block size grows with the pair
// triangle so that every thread owns at most `per` slots (8, or 12 where measured faster: 65-78 reads); the shared-memory footprint (two n x n int32 matrices) is
// sized by the class's largest n.
struct ClusterClass { int nmax, nt, per; };
static const ClusterClass kCluster[] = {{16, 32, 8}, {23, 32, 8}, {28, 64, 8}, {32, 64, 8}, {36, 96, 8}, {39, 96, 8}, {42, 128, 8}, {45, 128, 8},
                                    {50, 192, 8}, {55, 192, 8}, {60, 256, 8}, {64, 256, 8}, {71, 256, 12}, {78, 256, 12}, {85, 512, 8}, {91, 512, 8},
                                    {101, 768, 8}, {111, 768, 8}, {120, 1024, 8}, {128, 1024, 8},
                                    {136, 1024, 9}, {148, 1024, 11}, {160, 1024, 13}};
constexpr int N_CLUSTER = (int)(sizeof(kCluster) / sizeof(kCluster[0]));
// Scoring: (largest n, threads per block >= n, sort keys per lane)
struct ScoreClass { int nmax, nt, kpl; };
static const ScoreClass kScore[] = {{32, 64, 1}, {48, 128, 2}, {64, 128, 2}, {96, 256, 4}, {128, 256, 4}, {160, 256, 8}};
constexpr int N_SCORE = (int)(sizeof(kScore) / sizeof(kScore[0]));

#define AHS_FOR_EACH_NT(X) X(32, 8) X(64, 8) X(96, 8) X(128, 8) X(192, 8) X(256, 8) X(512, 8) X(768, 8) X(1024, 8) X(256, 12) X(1024, 9) X(1024, 11) X(1024, 13)
#define AHS_FOR_EACH_SC(X) X(64, 1) X(128, 2) X(256, 4) X(256, 8)
static void chain_kernel_attributes(size_t optin) {
#define X(NT, PER) CK(cudaFuncSetAttribute(k_cluster_chain<NT, PER>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)optin)); \
                   CK(cudaFuncSetAttribute(k_cluster_chain<NT, PER>, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    AHS_FOR_EACH_NT(X)
#undef X
#define X(NT, KPL) CK(cudaFuncSetAttribute(k_score_chain<2, NT, KPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)optin)); \
                   CK(cudaFuncSetAttribute(k_score_chain<4, NT, KPL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)optin));
    AHS_FOR_EACH_SC(X)
#undef X
}
static void cluster_launch(int nt, int per, unsigned grid, size_t smem, cudaStream_t st, const DB& d, const int32_t* list, int len, int nmax, int32_t* counter, int32_t* scratch) {
#define X(NT, PER) if (nt == NT && per == PER) { k_cluster_chain<NT, PER><<<grid, NT, smem, st>>>(d, list, len, nmax, counter, scratch); return; }
    AHS_FOR_EACH_NT(X)
#undef X
    throw ArgFail{"cluster_launch: no kernel for this block size"};
}
template <int BITS> static void score_launch(int nt, int kpl, unsigned grid, size_t smem, cudaStream_t st, const DB& d, const int32_t* list, int len, int nmax, int32_t* counter) {
#define X(NT, KPL) if (nt == NT && kpl == KPL) { k_score_chain<BITS, NT, KPL><<<grid, NT, smem, st>>>(d, list, len, nmax, counter); return; }
    AHS_FOR_EACH_SC(X)
#undef X
    throw ArgFail{"score_launch: no kernel for this block size"};
}
static int score_class(int n) { for (int k = 0; k < N_SCORE; k++) if (n <= kScore[k].nmax) return k; return -1; }
// every class must fit the device (checked once per context)
static void check_classes(size_t smem_optin) {
    for (int k = 0; k < N_CLUSTER; k++) {
        if (cc_smem_bytes(kCluster[k].nmax, kCluster[k].nt) > smem_optin) throw LimitFail{"device shared memory too small for the cluster-editing classes"};
        if ((int64_t)kCluster[k].nmax * (kCluster[k].nmax - 1) / 2 > (int64_t)kCluster[k].per * kCluster[k].nt) throw std::logic_error("cluster class table: slots");
        if (kCluster[k].nmax * cc_fresh_g(kCluster[k].nt, kCluster[k].per) > kCluster[k].nt) throw std::logic_error("cluster class table: fresh-cost lanes");
        if (kCluster[k].nmax > 128 && !(kCluster[k].nt == 1024 && kCluster[k].per > 8)) throw std::logic_error("cluster class table: classes above 128 reads need the five-stride kernels");
    }
    if (kCluster[N_CLUSTER - 1].nmax != CC_MAXN || kScore[N_SCORE - 1].nmax != CC_MAXN) throw std::logic_error("class tables do not end at CC_MAXN");
    for (int k = 0; k < N_SCORE; k++) if (kScore[k].nmax > kScore[k].nt || kScore[k].nmax > 32 * kScore[k].kpl || cs_smem_bytes(kScore[k].nmax, kScore[k].nt) > smem_optin) throw std::logic_error("score class table");
}

// neighbour tables of the sub-multiset lattice (k_thread_canon.cuh), built once per device
static void build_canon_tables(CanonTables& tb) {
    std::vector<uint32_t> tup; std::vector<uint16_t> add, del;
    for (int j = 0; j <= CN_P; j++) for (int k = 0; k <= CN_K; k++) tb.nn[j][k] = cn_count(j, k);
    tb.base[0] = 0;
    for (int k = 1; k <= CN_K; k++) {
        tb.base[k] = (int32_t)tup.size();
        int off = 0;
        for (int j = 0; j <= CN_P; j++) {
            tb.lvl[k][j] = off;
            const int cnt = cn_count(j, k);
            std::vector<int> x(j, 0);
            for (int e = 0; e < cnt; e++) {
                uint8_t t[CN_P + 1]; uint32_t packed = 0;
                for (int i = 0; i < j; i++) { t[i] = (uint8_t)x[i]; packed |= (uint32_t)x[i] << (4 * i); }
                if (cn_rank(t, j, k, tb.nn) != e) throw std::logic_error("canonical tuple tables: rank");
                tup.push_back(packed);
                for (int g = 0; g < 8; g++) {                  // insert g
                    uint16_t r = 0;
                    if (j < CN_P && g < k) {
                        uint8_t y[CN_P + 1]; int w = 0; bool done = false;
                        for (int i = 0; i < j; i++) { if (!done && g < t[i]) { y[w++] = (uint8_t)g; done = true; } y[w++] = t[i]; }
                        if (!done) y[w++] = (uint8_t)g;
                        r = (uint16_t)cn_rank(y, j + 1, k, tb.nn);
                    }
                    add.push_back(r);
                }
                for (int i = 0; i < 6; i++) {                  // delete element i
                    uint16_t r = 0;
                    if (i < j) { uint8_t y[CN_P + 1]; int w = 0; for (int u = 0; u < j; u++) if (u != i) y[w++] = t[u]; r = (uint16_t)cn_rank(y, j - 1, k, tb.nn); }
                    del.push_back(r);
                }
                // next non-decreasing tuple
                int i = j - 1;
                while (i >= 0 && x[i] == k - 1) i--;
                if (i >= 0) { const int v = x[i] + 1; for (int u = i; u < j; u++) x[u] = v; }
            }
            off += cnt;
        }
        tb.lvl[k][CN_P + 1] = off;
    }
    for (int j = 0; j <= CN_P + 1; j++) tb.lvl[0][j] = 0;
    uint32_t* d_tup; uint16_t *d_add, *d_del;
    CK(cudaMalloc(&d_tup, tup.size() * 4)); CK(cudaMalloc(&d_add, add.size() * 2)); CK(cudaMalloc(&d_del, del.size() * 2));
    CK(cudaMemcpy(d_tup, tup.data(), tup.size() * 4, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_add, add.data(), add.size() * 2, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(d_del, del.data(), del.size() * 2, cudaMemcpyHostToDevice));
    tb.tup = d_tup; tb.add = d_add; tb.del = d_del;
}

static Ctx* get_ctx(int device) {
    std::lock_guard<std::mutex> g(g_ctx_mu);
    if (device < 0 || device >= 64) throw ArgFail{"device ordinal out of range"};
    if (g_ctx[device]) return g_ctx[device];
    int n = 0; CK(cudaGetDeviceCount(&n));
    if (device >= n) throw ArgFail{"no such CUDA device"};
    CK(cudaSetDevice(device));
    Ctx* c = new Ctx(); c->device = device;
    for (auto& ln : c->lanes) {
        CK(cudaStreamCreateWithFlags(&ln.stream, cudaStreamNonBlocking));
        CK(cudaStreamCreateWithFlags(&ln.stream2, cudaStreamNonBlocking));
        for (auto& e : ln.ev) CK(cudaEventCreate(&e));
        CK(cudaEventCreateWithFlags(&ln.ev_cells, cudaEventDisableTiming));
        for (auto& e : ln.ev_en) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
        CK(cudaEventCreateWithFlags(&ln.ev_fork, cudaEventDisableTiming));
        CK(cudaEventCreate(&ln.ev_up));
        for (auto& e : ln.ev_join) CK(cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    }
    for (auto& t : c->side) CK(cudaStreamCreateWithFlags(&t, cudaStreamNonBlocking));
    cudaDeviceProp prop; CK(cudaGetDeviceProperties(&prop, device)); c->sms = prop.multiProcessorCount;
    // fixed-point log tables of rule R1 (oracle/core/phase_core.hpp): llrint(ln(x/1024) * 2^20)
    std::vector<int64_t> ln(1025, 0), ln1(1025, 0);
    for (int x = 0; x <= 1024; x++) {
        if (x >= 1) ln[x] = llrint(std::log((double)x / 1024.0) * 1048576.0);
        if (x <= 1023) ln1[x] = llrint(std::log(1.0 - (double)x / 1024.0) * 1048576.0);
    }
    CK(cudaMalloc(&c->d_ln, 1025 * 8)); CK(cudaMalloc(&c->d_ln1, 1025 * 8));
    CK(cudaMemcpy(c->d_ln, ln.data(), 1025 * 8, cudaMemcpyHostToDevice));
    CK(cudaMemcpy(c->d_ln1, ln1.data(), 1025 * 8, cudaMemcpyHostToDevice));
    CK(cudaFuncSetAttribute(k_thread, cudaFuncAttributeMaxDynamicSharedMemorySize, 21 * 4096 + 64));
    CK(cudaFuncSetAttribute(k_thread_canon<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    CK(cudaFuncSetAttribute(k_thread_canon<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
    CK(cudaFuncSetAttribute(k_chain_front, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FR_SMEM_CAP));
    build_canon_tables(c->canon);
    c->smem_optin = prop.sharedMemPerBlockOptin;
    check_classes(c->smem_optin);
    CK(cudaFuncSetAttribute(k_cluster_sparse<SP_THREADS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_optin));
    CK(cudaFuncSetAttribute(k_cluster_sparse<SP_THREADS_SMALL>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)c->smem_optin));
    chain_kernel_attributes(c->smem_optin);
    g_ctx[device] = c;
    return c;
}

// ------------------------------------------------------------------ validation
struct Sizes { int64_t C, NB, NA, NAN_, NR, NE, NEN, M; int max_k; };

// Host side: O(chains) checks only.  Everything per bubble / allele / entry is checked on the device by
// k_validate* (first kernels of the pass) and reported after sync #1.
static Sizes validate(const ahs_batch_in* in, bool is_view = false) {
    if (!in) throw ArgFail{"null batch"};
    if (in->n_chains < 0) throw ArgFail{"n_chains < 0"};
    if (in->ploidy < 1 || in->ploidy > MAX_PLOIDY) throw LimitFail{"ploidy outside [1," + std::to_string(MAX_PLOIDY) + "]"};
    Sizes s{}; s.C = in->n_chains;
    if (s.C == 0) return s;
    auto mono = [&](const int64_t* off, int64_t n, const char* name) {
        if (!off) throw ArgFail{std::string(name) + " is null"};
        if (off[0] != 0) throw ArgFail{std::string(name) + "[0] != 0"};
        for (int64_t i = 0; i < n; i++) if (off[i + 1] < off[i]) throw ArgFail{std::string(name) + " not monotone"};
    };
    auto ends = [&](const int64_t* off, int64_t n, const char* name) -> int64_t {      // a view (chunk of chains) starts at its base
        if (!off) throw ArgFail{std::string(name) + " is null"};
        if (!is_view && off[0] != 0) throw ArgFail{std::string(name) + "[0] != 0"};
        if (off[n] < off[0]) throw ArgFail{std::string(name) + " not monotone"};
        return off[n] - off[0];
    };
    mono(in->bubble_off, s.C, "bubble_off"); s.NB = in->bubble_off[s.C];
    s.NA = ends(in->allele_off, s.NB, "allele_off");
    s.NAN_ = ends(in->anode_off, s.NA, "anode_off");
    mono(in->read_off, s.C, "read_off"); s.NR = in->read_off[s.C];
    mono(in->entry_off, s.C, "entry_off"); s.NE = in->entry_off[s.C];
    s.NEN = ends(in->enode_off, s.NE, "enode_off");
    if ((s.NAN_ && !in->anode) || (s.NEN && !in->enode) || (s.NE && (!in->entry_read || !in->entry_identity))) throw ArgFail{"null array"};
    for (int64_t c = 0; c < s.C; c++) {
        const int64_t B = in->bubble_off[c + 1] - in->bubble_off[c], R = in->read_off[c + 1] - in->read_off[c];
        if (B > MAX_POSITIONS) throw LimitFail{"chain with more than 32767 bubbles"};
        if (R > MAX_READS_CHAIN) throw LimitFail{"chain with more than 2^20 distinct read names (the read order is ranked by pairwise counting)"};
        s.M += (B > 1) ? B * R : 0;
    }
    s.max_k = 0;                                     // filled in from the device at sync #1
    return s;
}

__global__ void k_fetch_host(const int4* __restrict__ src, int4* __restrict__ dst, int64_t n) {
    for (int64_t i = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; i < n; i += (int64_t)gridDim.x * blockDim.x) dst[i] = src[i];
}

static inline int grid_for(int64_t items, int per_block, int sms) {
    int64_t g = (items + per_block - 1) / per_block;
    int64_t cap = (int64_t)sms * 16;
    return (int)std::max<int64_t>(1, std::min(g, cap));
}

// ------------------------------------------------------------------ the pipeline
struct Pipeline {
    Ctx* cx; Lane* ln; const ahs_batch_in* in; Sizes sz; DB d{};
    const uint8_t* dosage = nullptr;                                            // caller genotypes of `in` (indexed like its allele_off), or null
    std::vector<int64_t> h_mrow_off, h_frow_off, h_pos_off, h_code_off, h_cw_off, h_back_off;
    int32_t *h_status = nullptr, *h_nfinal = nullptr, *h_npos = nullptr;      // pinned: D2H targets of sync #1
    int64_t* h_sc = nullptr;                                                   // pinned scalars of sync #1: cells, error flags, largest allele count
    unsigned long long* h_cells = nullptr;
    char *sg_h = nullptr, *sg_d = nullptr; size_t sg_cap = 0;                   // pinned / device staging block of phase 2
    bool early_out = false;                                                     // download the matrix while the clustering runs
    int64_t base_allele = 0, base_anode = 0, base_enode = 0;                    // first elements of the three big offset arrays (chunk views)
    int64_t cell_base = 0;                                                      // cells of the chunks before this one (cell_off is global)
    static constexpr int N_EN = 6; int64_t en_cut[N_EN + 1] = {0};              // entry ranges whose alignment nodes are uploaded as one slice
    int64_t n_code_words = 0, n_cw = 0, h_tot_cells = 0, h_slots = 0;
    size_t front_smem = 0; bool use_front = false;                              // one block per chain for projection + rows (k_front.cuh)
    std::vector<uint32_t> front_need;                                           // per chain: shared memory of its block
    float ms[7] = {0};
    int n_launches = 0;

    template <class T> const T* up(const T* h, int64_t n) {
        T* p = cx->dev.get<T>((size_t)std::max<int64_t>(n, 1));
        if (n > 0) CK(cudaMemcpyAsync(p, h, n * sizeof(T), cudaMemcpyHostToDevice, ln->stream));
        return p;
    }
    // host-derived arrays go through pinned staging: an async copy from pageable memory would first drain the stream
    template <class T> const T* up_pinned(const T* h, int64_t n) {
        T* stage = cx->pin.get<T>((size_t)std::max<int64_t>(n, 1));
        if (n > 0) memcpy(stage, h, n * sizeof(T));
        return up(stage, n);
    }
    template <class T> T* dalloc(int64_t n) { return cx->dev.get<T>((size_t)std::max<int64_t>(n, 1)); }
    template <class T> T* dzero(int64_t n) { T* p = dalloc<T>(n); CK(cudaMemsetAsync(p, 0, std::max<int64_t>(n, 1) * sizeof(T), ln->stream)); return p; }
    template <class T> T* dfill_ff(int64_t n) { T* p = dalloc<T>(n); CK(cudaMemsetAsync(p, 0xff, std::max<int64_t>(n, 1) * sizeof(T), ln->stream)); return p; }

    // `after`: lane whose upload must be through first — uploads of successive ranges share the copy engines, and run one
    // after the other so that the first range is complete (and its projection starts) as early as possible
    void upload(Lane* after = nullptr) {
        cudaStream_t st = ln->stream;
        const int64_t C = sz.C;
        if (after && after != ln) { CK(cudaStreamWaitEvent(ln->stream, after->ev_up, 0)); CK(cudaStreamWaitEvent(ln->stream2, after->ev_up, 0)); }
        d.C = (int32_t)C; d.ploidy = in->ploidy; d.bits = 2;      // code width is decided at sync #1 (largest allele count)
        d.NB = sz.NB; d.NA = sz.NA; d.NAN_ = sz.NAN_; d.NR = sz.NR; d.NE = sz.NE; d.NEN = sz.NEN;
        d.bubble_off = up(in->bubble_off, C + 1); d.allele_off = up(in->allele_off, sz.NB + 1); d.anode_off = up(in->anode_off, sz.NA + 1);
        d.read_off = up(in->read_off, C + 1); d.entry_off = up(in->entry_off, C + 1); d.enode_off = up(in->enode_off, sz.NE + 1);
        base_allele = in->allele_off[0]; base_anode = in->anode_off[0]; base_enode = in->enode_off[0];
        // the alignment nodes are 3/4 of the batch: they go up in N_EN slices on the second stream, and the projection of
        // slice i runs under the upload of slice i+1
        base_enode = in->enode_off[0];
        {
            int32_t* en = cx->dev.get<int32_t>((size_t)std::max<int64_t>(sz.NEN, 1));
            d.enode = en;
            for (int i = 0; i <= N_EN; i++) {
                const int64_t target = base_enode + sz.NEN / N_EN * i;
                en_cut[i] = i == N_EN ? sz.NE : (int64_t)(std::lower_bound(in->enode_off, in->enode_off + sz.NE, target) - in->enode_off);
            }
            en_cut[0] = 0;
            for (int i = 0; i < N_EN; i++) {
                en_cut[i + 1] = std::max(en_cut[i + 1], en_cut[i]);
                const int64_t o0 = std::min<int64_t>(std::max<int64_t>(in->enode_off[en_cut[i]] - base_enode, 0), sz.NEN);
                const int64_t o1 = i + 1 == N_EN ? sz.NEN : std::min<int64_t>(std::max<int64_t>(in->enode_off[en_cut[i + 1]] - base_enode, o0), sz.NEN);
                if (o1 > o0) CK(cudaMemcpyAsync(en + o0, in->enode + o0, (size_t)(o1 - o0) * 4, cudaMemcpyHostToDevice, ln->stream2));
                CK(cudaEventRecord(ln->ev_en[i], ln->stream2));
            }
        }
        d.anode = up(in->anode, sz.NAN_); d.entry_read = up(in->entry_read, sz.NE);
        d.entry_identity = up(in->entry_identity, sz.NE);
        d.stage_a_order = in->stage_a_order ? up(in->stage_a_order, sz.NB) : nullptr;
        d.allele_dosage = dosage ? up(dosage, sz.NA) : nullptr;
        h_mrow_off.assign(C, 0);
        int64_t acc = 0;
        for (int64_t c = 0; c < C; c++) {
            h_mrow_off[c] = acc;
            const int64_t B = in->bubble_off[c + 1] - in->bubble_off[c], R = in->read_off[c + 1] - in->read_off[c];
            if (B > 1) acc += B * R;
            if (acc & 1) acc++;                                    // keep chain bases 4-byte aligned for the 32-bit atomics
        }
        sz.M = acc;
        d.mrow_off = (int64_t*)up_pinned(h_mrow_off.data(), C);
        // per-chain trigger tables: power of two >= 4 x alleles of the chain (most probes are misses: they end at the first empty slot)
        std::vector<int64_t> hoff(C); std::vector<uint32_t> hmaskc(C);
        h_slots = 0; front_need.assign(C, 0); front_smem = 0;
        for (int64_t c = 0; c < C; c++) {
            const int64_t nal = in->allele_off[in->bubble_off[c + 1]] - in->allele_off[in->bubble_off[c]];
            if (nal < 0 || nal > sz.NA) throw ArgFail{"allele_off / anode_off / enode_off not monotone"};
            int64_t cap = 4; while (cap < 4 * nal) cap <<= 1;
            hoff[c] = h_slots; hmaskc[c] = (uint32_t)(cap - 1); h_slots += cap;
            const int64_t B = in->bubble_off[c + 1] - in->bubble_off[c], R = in->read_off[c + 1] - in->read_off[c], NEc = in->entry_off[c + 1] - in->entry_off[c];
            const int64_t e_lo = in->entry_off[c], e_hi = in->entry_off[c + 1];
            if (e_lo < 0 || e_hi < e_lo || e_hi > sz.NE) throw ArgFail{"entry_off out of range"};
            const int64_t NENc = in->enode_off[e_hi] - in->enode_off[e_lo];
            if (B > 1) {
                if (NENc < 0 || NENc > sz.NEN || R * B > ((int64_t)1 << 24) || cap > (1 << 20)) front_smem = SIZE_MAX / 2;
                else { front_need[c] = fr_layout((int)B, (int)R, (int)nal, (int)NEc, (int)NENc, (int)cap).total; front_smem = std::max(front_smem, (size_t)front_need[c]); }
            }
        }
        use_front = front_smem <= FR_SMEM_CAP;
        d.hoff = up_pinned(hoff.data(), C); d.hmaskc = up_pinned(hmaskc.data(), C);
        CK(cudaStreamWaitEvent(st, ln->ev_en[N_EN - 1], 0));
        CK(cudaEventRecord(ln->ev_up, st));                    // the copies are through: the next range's may start
        // a view's interior offsets are rebased on the device — after the event, so that a kernel waiting for a free SM never holds up a copy
        if (base_allele) k_rebase<<<grid_for(sz.NB + 1, 256, cx->sms), 256, 0, st>>>((int64_t*)d.allele_off, sz.NB + 1, base_allele);
        if (base_anode) k_rebase<<<grid_for(sz.NA + 1, 256, cx->sms), 256, 0, st>>>((int64_t*)d.anode_off, sz.NA + 1, base_anode);
        if (base_enode) k_rebase<<<grid_for(sz.NE + 1, 256, cx->sms), 256, 0, st>>>((int64_t*)d.enode_off, sz.NE + 1, base_enode);
    }

    // allocate and initialise everything phase 1 writes; called once per run (also per resident iteration)
    void alloc_phase1() {
        const int64_t C = sz.C;
        d.bubble_chain = dalloc<int32_t>(sz.NB); d.allele_bubble = dalloc<int32_t>(sz.NA); d.entry_chain = dalloc<int32_t>(sz.NE);
        d.read_chain = dalloc<int32_t>(sz.NR); d.rankA = dalloc<int32_t>(sz.NB);
        d.hslots = dalloc<unsigned long long>(h_slots); d.inc_next = dalloc<int32_t>(sz.NA); d.arec = dalloc<int4>(sz.NA);
        d.bubble_univ = dalloc<uint32_t>(sz.NB);
        d.mask = dalloc<uint16_t>(sz.M + 2);
        d.create_key = dalloc<uint64_t>(sz.NR); d.createA_key = dalloc<uint64_t>(sz.NR); d.first_entry = dalloc<uint32_t>(sz.NR);
        d.has_good = dalloc<uint8_t>(sz.NR);
        d.rdA_cnt = dalloc<int32_t>(sz.NR); d.rdA_first = dalloc<int32_t>(sz.NR); d.rdA_last = dalloc<int32_t>(sz.NR); d.rdA_mapq = dalloc<int32_t>(sz.NR);
        d.rd_nv = dalloc<int32_t>(sz.NR); d.rd_first = dalloc<int32_t>(sz.NR); d.rd_last = dalloc<int32_t>(sz.NR); d.rd_mapq = dalloc<int32_t>(sz.NR);
        d.rd_pass = dalloc<uint8_t>(sz.NR); d.ord = dalloc<int32_t>(sz.NR); d.okey = dalloc<int32_t>(sz.NR);
        d.poscov = dalloc<uint8_t>(sz.NB); d.pos_compact = dalloc<int32_t>(sz.NB);
        d.ch_status = dalloc<int32_t>(C); d.ch_maxpos = dalloc<int32_t>(C); d.ch_flags = dalloc<int32_t>(C); d.ch_T = dalloc<int32_t>(C);
        d.ch_nfinal = dalloc<int32_t>(C); d.ch_npos = dalloc<int32_t>(C); d.ch_maxspan = dalloc<int32_t>(C); d.ch_words = dalloc<int32_t>(C);
        d.ch_nclusters = dalloc<int32_t>(C); d.ch_cells = dalloc<unsigned long long>(C); d.ch_pairs2 = dalloc<unsigned long long>(C);
        d.tot_cells = dalloc<int64_t>(1); d.tot_pairs = dalloc<int64_t>(1); d.err_flags = dalloc<int32_t>(1);
        d.ln = cx->d_ln; d.ln1 = cx->d_ln1;
        h_status = cx->pin.get<int32_t>(C); h_nfinal = cx->pin.get<int32_t>(C); h_npos = cx->pin.get<int32_t>(C); h_sc = cx->pin.get<int64_t>(4);
        h_cells = cx->pin.get<unsigned long long>(C);
        sg_cap = (size_t)(C + 2) * (8 * 5 + 4 * 3 + 1) + 512;
        sg_h = (char*)cx->pin.alloc(sg_cap); sg_d = (char*)cx->dev.alloc(sg_cap);
    }

    void init_phase1() {
        cudaStream_t st = ln->stream; const int64_t C = sz.C;
        CK(cudaMemsetAsync(d.hslots, 0xff, (size_t)std::max<int64_t>(h_slots, 1) * 8, st));
        CK(cudaMemsetAsync(d.bubble_univ, 0xff, std::max<int64_t>(sz.NB, 1) * 4, st));
        CK(cudaMemsetAsync(d.mask, 0, (sz.M + 2) * 2, st));
        CK(cudaMemsetAsync(d.create_key, 0xff, std::max<int64_t>(sz.NR, 1) * 8, st)); CK(cudaMemsetAsync(d.createA_key, 0xff, std::max<int64_t>(sz.NR, 1) * 8, st));
        CK(cudaMemsetAsync(d.first_entry, 0xff, std::max<int64_t>(sz.NR, 1) * 4, st)); CK(cudaMemsetAsync(d.has_good, 0, std::max<int64_t>(sz.NR, 1), st));
        CK(cudaMemsetAsync(d.poscov, 0, std::max<int64_t>(sz.NB, 1), st));
        CK(cudaMemsetAsync(d.rankA, 0xff, std::max<int64_t>(sz.NB, 1) * 4, st));
        CK(cudaMemsetAsync(d.ch_status, 0, C * 4, st)); CK(cudaMemsetAsync(d.ch_maxpos, 0xff, C * 4, st)); CK(cudaMemsetAsync(d.ch_flags, 0, C * 4, st));
        CK(cudaMemsetAsync(d.ch_nfinal, 0, C * 4, st)); CK(cudaMemsetAsync(d.ch_maxspan, 0, C * 4, st)); CK(cudaMemsetAsync(d.ch_nclusters, 0, C * 4, st));
        CK(cudaMemsetAsync(d.ch_cells, 0, C * 8, st)); CK(cudaMemsetAsync(d.ch_pairs2, 0, C * 8, st));
        CK(cudaMemsetAsync(d.tot_cells, 0, 8, st)); CK(cudaMemsetAsync(d.tot_pairs, 0, 8, st)); CK(cudaMemsetAsync(d.err_flags, 0, 4, st));
    }

    void scan(const int32_t* in32, int64_t n, int64_t* out, int64_t base) {       // out[n+1] = base + exclusive prefix sums
        cudaStream_t st = ln->stream;
        const int64_t nb = std::max<int64_t>(1, (n + SCAN_BLOCK - 1) / SCAN_BLOCK);
        int64_t* bs = dalloc<int64_t>(nb + 1);
        k_scan_local<<<(unsigned)nb, SCAN_BLOCK, 0, st>>>(in32, n, out, bs); n_launches += 1;
        k_scan_blocks<<<1, SCAN_BLOCK, 0, st>>>(bs, nb, bs + nb); n_launches += 1;
        k_scan_add<<<(unsigned)nb, SCAN_BLOCK, 0, st>>>(out, n, bs, bs + nb, base); n_launches += 1;
        CK(cudaGetLastError());
    }

    // phase 1: validation, projection, final rows per read, read order — enqueued, with the copies of sync #1 behind it
    void run_phase1_enqueue() {
        cudaStream_t st = ln->stream; const int sms = cx->sms; const int64_t C = sz.C;
        const int TB = 256;
        n_launches = 0;
        CK(cudaEventRecord(ln->ev[0], st));
        init_phase1();
        int32_t* d_maxk = dzero<int32_t>(1);
        k_validate<<<grid_for(std::max(sz.NE, std::max(sz.NA, sz.NB)), TB, sms), TB, 0, st>>>(d, d_maxk); n_launches += 1;
        if (use_front) {
            // every chain's working set fits a block's shared memory: projection, stage A / B, filter and read order in ONE
            // kernel, one block per chain (k_front.cuh); the chain's alignment nodes arrive by a bulk asynchronous copy
            for (int i = 0; i < N_EN; i++) CK(cudaStreamWaitEvent(st, ln->ev_en[i], 0));
            // ranges of chains by shared-memory need (more resident blocks for the many small chains): cut where the largest need of
            // the remaining chains falls below a threshold
            std::vector<uint32_t> sufmax(C + 1, 0);
            for (int64_t c = C - 1; c >= 0; c--) sufmax[c] = std::max(sufmax[c + 1], front_need[c]);
            int32_t* fcount = dzero<int32_t>(4);
            int64_t c_begin = 0; int seg = 0;
            for (uint32_t thr : {54u << 10, 26u << 10, 12u << 10, 0u}) {
                int64_t c_end = C;
                if (thr) { c_end = c_begin; while (c_end < C && sufmax[c_end] > thr) c_end++; }       // first chain from which everything fits `thr`
                if (c_end > c_begin) {
                    const size_t smem = std::max<size_t>(sufmax[c_begin], 1024);
                    const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (220 * 1024) / (smem + 1024)));
                    k_chain_front<<<(unsigned)std::min<int64_t>(c_end - c_begin, (int64_t)sms * per_sm), FR_THREADS, smem, st>>>(d, (int)c_begin, (int)c_end, fcount + seg);
                    n_launches += 1;
                }
                c_begin = c_end; seg++;
                if (c_begin >= C) break;
            }
            CK(cudaEventRecord(ln->ev[1], st));
        } else {
            // ---- owner maps + trigger table
            if (sz.NB) k_owner<<<grid_for(sz.NB, TB, sms), TB, 0, st>>>(d.bubble_off, (int)C, sz.NB, d.bubble_chain); n_launches += 1;
            if (sz.NA) k_owner<<<grid_for(sz.NA, TB, sms), TB, 0, st>>>(d.allele_off, (int)sz.NB, sz.NA, d.allele_bubble); n_launches += 1;
            if (sz.NE) k_owner<<<grid_for(sz.NE, TB, sms), TB, 0, st>>>(d.entry_off, (int)C, sz.NE, d.entry_chain); n_launches += 1;
            if (sz.NR) k_owner<<<grid_for(sz.NR, TB, sms), TB, 0, st>>>(d.read_off, (int)C, sz.NR, d.read_chain); n_launches += 1;
            k_validate_owned<<<grid_for(sz.NE, TB, sms), TB, 0, st>>>(d); n_launches += 1;
            if (sz.NB) k_rank_a<<<grid_for(sz.NB, TB, sms), TB, 0, st>>>(d); n_launches += 1;
            if (sz.NB && d.stage_a_order) { k_validate_perm<<<grid_for(sz.NB, TB, sms), TB, 0, st>>>(d); n_launches += 1; }
            if (sz.NA) k_build_triggers<<<grid_for(sz.NA, TB, sms), TB, 0, st>>>(d); n_launches += 1;
            // ---- projection
            for (int i = 0; i < N_EN; i++) {
                CK(cudaStreamWaitEvent(st, ln->ev_en[i], 0));
                const int64_t ne = en_cut[i + 1] - en_cut[i];
                if (ne > 0) {
                    if (sz.NEN <= 48 * sz.NE) k_project<16><<<grid_for(ne, 16, sms), TB, 0, st>>>(d, en_cut[i], en_cut[i + 1]);      // short alignments
                    else k_project<32><<<grid_for(ne, 8, sms), TB, 0, st>>>(d, en_cut[i], en_cut[i + 1]);
                    n_launches += 1;
                }
            }
            CK(cudaEventRecord(ln->ev[1], st));
            const bool small_rows = sz.NB <= 96 * C;        // short chains: 8 lanes per read, 4 reads in flight per warp
            if (sz.NR) { if (small_rows) k_read_stage_a<8><<<grid_for(sz.NR, 32, sms), TB, 0, st>>>(d); else k_read_stage_a<32><<<grid_for(sz.NR, 8, sms), TB, 0, st>>>(d); n_launches += 1; }
            if (sz.NR) k_chain_flags<<<grid_for(sz.NR, TB, sms), TB, 0, st>>>(d); n_launches += 1;
            k_chain_T<<<grid_for(C, TB, sms), TB, 0, st>>>(d); n_launches += 1;
            if (sz.NR) { if (small_rows) k_read_rows<8><<<grid_for(sz.NR, 32, sms), TB, 0, st>>>(d); else k_read_rows<32><<<grid_for(sz.NR, 8, sms), TB, 0, st>>>(d); n_launches += 1; }
            if (sz.NR) k_read_rank<<<grid_for(sz.NR, TB, sms), TB, 0, st>>>(d); n_launches += 1;
            k_chain_sort<<<grid_for(C, 64, sms), 64, 0, st>>>(d); n_launches += 1;
            k_count_pos<<<grid_for(C, 8, sms), TB, 0, st>>>(d); n_launches += 1;
        }
        CK(cudaGetLastError());
        // ---- sync #1: per-chain sizes -> offsets of the per-chain workspaces
        h_sc[0] = 0; h_sc[1] = 0; h_sc[2] = 0;
        CK(cudaMemcpyAsync(h_status, d.ch_status, C * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(h_nfinal, d.ch_nfinal, C * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(h_npos, d.ch_npos, C * 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(h_cells, d.ch_cells, C * 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&h_sc[0], d.tot_cells, 8, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&h_sc[1], d.err_flags, 4, cudaMemcpyDeviceToHost, st));
        CK(cudaMemcpyAsync(&h_sc[2], d_maxk, 4, cudaMemcpyDeviceToHost, st));
    }
    // sync #1: per-chain sizes on the host
    void run_phase1_finish() {
        CK(cudaStreamSynchronize(ln->stream));
        h_tot_cells = h_sc[0];
        const int32_t h_err = (int32_t)h_sc[1], h_maxk = (int32_t)h_sc[2];
        if (h_err & 4) throw ArgFail{"allele_off / anode_off / enode_off not monotone"};
        if (h_err & 1) throw ArgFail{"empty allele path"};
        if (h_err & 2) throw LimitFail{"a bubble has more than 15 alleles"};
        if (h_err & 8) throw ArgFail{"entry_read out of range"};
        if (h_err & 16) throw ArgFail{"stage_a_order is not a permutation"};
        if (h_err & 32) throw ArgFail{"allele_dosage: the dosages of a bubble are neither all 0 nor sum to the ploidy"};
        sz.max_k = h_maxk;
        d.bits = sz.max_k <= 3 ? 2 : 4;
    }

    // pinned staging block: every per-chain array the host derives at sync #1 goes to the device in ONE copy
    struct Stage {
        char* h = nullptr; char* dv = nullptr; size_t used = 0;
        template <class T> T* take(size_t n, T** dev) { used = (used + 15) & ~(size_t)15; T* p = (T*)(h + used); *dev = (T*)(dv + used); used += n * sizeof(T); return p; }
    };

    template <int BITS> void run_bits() {
        cudaStream_t st = ln->stream; const int sms = cx->sms; const int64_t C = sz.C;
        const int TB = 256;
        const int per_word = 32 / BITS;
        int64_t S_max = 1; for (int i = 0; i < in->ploidy; i++) S_max *= 2 * in->ploidy;
        if (in->ploidy > 4) S_max = cn_count(in->ploidy, in->ploidy + 2);      // canonical tuples over p + 2 clusters (rule R3c)
        d.S_max = (int32_t)S_max;
        Stage sg; sg.h = sg_h; sg.dv = sg_d;
        int64_t *dv_frow, *dv_pos, *dv_code, *dv_cw, *dv_back; int32_t *dv_words, *dv_order, *dv_status; uint8_t* dv_small;
        int64_t* s_frow = sg.take<int64_t>(C + 1, &dv_frow); int64_t* s_pos = sg.take<int64_t>(C + 1, &dv_pos);
        int64_t* s_code = sg.take<int64_t>(C, &dv_code); int64_t* s_cw = sg.take<int64_t>(C, &dv_cw); int64_t* s_back = sg.take<int64_t>(C, &dv_back);
        int32_t* s_words = sg.take<int32_t>(C, &dv_words); int32_t* s_order = sg.take<int32_t>(C, &dv_order); int32_t* s_status = sg.take<int32_t>(C, &dv_status);
        uint8_t* s_small = sg.take<uint8_t>(C, &dv_small);
        if (sg.used > sg_cap) throw std::runtime_error("staging block overflow");
        n_code_words = 0; n_cw = 0;
        bool status_changed = false;
        s_frow[0] = 0; s_pos[0] = 0;
        int64_t nf_big = 0, cells_ok = 0; int n_max = 0;
        // chains above CC_MAXN reads take k_cluster_sparse (edge slots + lists)
        int max_reads = MAX_READS_CLUSTER;
        int64_t nf_sparse = 0;
        if (const char* e = getenv("AHS_MAX_READS_CLUSTER")) max_reads = std::max(CC_MAXN, std::min(max_reads, atoi(e)));      // tests: exercise the limit cheaply
        int64_t big_w_bytes = 0;
        for (int64_t c = 0; c < C; c++) {
            if (h_status[c] == AHS_CHAIN_OK && h_nfinal[c] > CC_MAXN) {
                // chains above the shared-memory kernels keep a dense n x n weight matrix in HBM: bounded per chain and per call
                const int64_t wb = (int64_t)h_nfinal[c] * h_nfinal[c] * 4;
                if (h_nfinal[c] > max_reads || big_w_bytes + wb > MAX_BIG_W_BYTES) { h_status[c] = AHS_CHAIN_TOO_LARGE; status_changed = true; }
                else big_w_bytes += wb;
            }
            s_status[c] = h_status[c];
            const bool ok = h_status[c] == AHS_CHAIN_OK;
            const int64_t n = ok ? h_nfinal[c] : 0, np = ok ? h_npos[c] : 0;
            h_nfinal[c] = (int32_t)n;
            const int64_t B = in->bubble_off[c + 1] - in->bubble_off[c];
            s_words[c] = (int32_t)((B + per_word - 1) / per_word);
            s_frow[c + 1] = s_frow[c] + n; s_pos[c + 1] = s_pos[c] + np;
            s_code[c] = n_code_words; n_code_words += n * s_words[c];
            s_small[c] = (n > 0 && n <= CC_MAXN) ? 1 : 0;
            s_cw[c] = n_cw; n_cw += s_small[c] ? n * (n - 1) / 2 : n * n;
            if (n > CC_MAXN) nf_sparse += n;
            s_back[c] = s_pos[c] * S_max;
            if (!s_small[c]) nf_big += n;
            n_max = std::max<int>(n_max, (int)n);
            if (ok) cells_ok += (int64_t)h_cells[c];
        }
        h_tot_cells = cells_ok;                            // chains dropped above (too many reads) emit nothing
        // chains by decreasing read count (counting sort): every size class is one contiguous range of `order`
        std::vector<int32_t> start(n_max + 2, 0);
        for (int64_t c = 0; c < C; c++) start[n_max - h_nfinal[c] + 1]++;
        for (int x = 0; x <= n_max; x++) start[x + 1] += start[x];
        { std::vector<int32_t> fill(start.begin(), start.end() - 1); for (int64_t c = 0; c < C; c++) s_order[fill[n_max - h_nfinal[c]]++] = (int32_t)c; }
        auto range_of = [&](int n_lo, int n_hi, int& first, int& len) {          // chains with n_lo <= n <= n_hi
            n_hi = std::min(n_hi, n_max); n_lo = std::max(n_lo, 0);
            if (n_hi < n_lo) { first = 0; len = 0; return; }
            first = start[n_max - n_hi]; len = start[n_max - n_lo + 1] - first;
        };
        h_frow_off.assign(s_frow, s_frow + C + 1); h_pos_off.assign(s_pos, s_pos + C + 1);
        const int64_t NF = s_frow[C], NP = s_pos[C];
        d.NF = NF; d.NP = NP;
        // the staging block is fetched by a kernel straight from page-locked host memory: a copy-engine transfer would queue behind the
        // bulk upload of the next range
        { const int64_t n16 = (int64_t)((sg.used + 15) / 16); k_fetch_host<<<grid_for(n16, 256, sms), 256, 0, st>>>((const int4*)sg.h, (int4*)sg.dv, n16); n_launches += 1; }
        d.frow_off = dv_frow; d.pos_off = dv_pos; d.code_off = dv_code; d.cw_off = dv_cw; d.back_off = dv_back;
        d.ch_words = dv_words; d.ch_small = dv_small;
        if (status_changed) CK(cudaMemcpyAsync(d.ch_status, dv_status, C * 4, cudaMemcpyDeviceToDevice, st));
        d.fr_chain = dalloc<int32_t>(NF); d.fr_first = dalloc<int32_t>(NF); d.fr_last = dalloc<int32_t>(NF); d.fr_mapq = dalloc<int32_t>(NF);
        d.fr_id = dalloc<int32_t>(NF); d.fr_nv = dalloc<int32_t>(NF); d.fr_cluster = dzero<int32_t>(NF);
        d.codes = dzero<uint32_t>(n_code_words);
        d.pos = dalloc<int32_t>(NP); d.pos_chain = dalloc<int32_t>(NP);
        d.es = dalloc<uint16_t>(NF); d.ed = dalloc<uint16_t>(NF);
        d.W = dalloc<int32_t>(n_cw);
        if (nf_big) {
            // HBM-resident path (chains above CC_MAXN reads): a dense n x n weight matrix per chain
            for (int64_t c = 0; c < C; c++) if (!s_small[c] && h_nfinal[c] > 0)
                CK(cudaMemsetAsync(d.W + s_cw[c], 0, (size_t)h_nfinal[c] * h_nfinal[c] * 4, st));
        }
        d.rec = dalloc<PosRec>(NP); d.back = dalloc<uint16_t>(NP * S_max);
        d.path = dzero<int32_t>(NP * in->ploidy); d.hap_allele = dzero<uint8_t>(NP * in->ploidy); d.dp_cost = dzero<double>(C);
        d.cell_off = dalloc<int64_t>(NF + 1); d.cell_pos = dalloc<int32_t>(h_tot_cells); d.cell_allele = dalloc<uint8_t>(h_tot_cells);
        int32_t* counters = dzero<int32_t>(8 + N_SCORE + N_CLUSTER);
        d.key_scratch = nullptr; d.key_scratch_off = nullptr;
        if (nf_big) {
            // reads of HBM-path chains with more than RATE_SMEM_KEYS candidate partners sort in HBM scratch
            std::vector<int64_t> koff(NF + 1, 0);
            int64_t tot = 0; bool any = false;
            for (int64_t c = 0; c < C; c++) {
                const int64_t n = h_nfinal[c];
                int64_t cap = 0;
                if (n > RATE_SMEM_KEYS && !s_small[c]) { cap = 1; while (cap < n) cap <<= 1; any = true; }
                for (int64_t i = 0; i < n; i++) { koff[s_frow[c] + i] = tot; tot += cap; }
            }
            koff[NF] = tot;
            if (any) { d.key_scratch = dalloc<uint64_t>(tot); d.key_scratch_off = (int64_t*)up(koff.data(), NF + 1); }
        }
        if (NF) k_owner<<<grid_for(NF, TB, sms), TB, 0, st>>>(d.frow_off, (int)C, NF, d.fr_chain); n_launches += 1;
        if (NP) k_owner<<<grid_for(NP, TB, sms), TB, 0, st>>>(d.pos_off, (int)C, NP, d.pos_chain); n_launches += 1;
        if (NF) { if (sz.NB <= 96 * C) k_pack_rows<8><<<grid_for(NF, 32, sms), TB, 0, st>>>(d); else k_pack_rows<32><<<grid_for(NF, 8, sms), TB, 0, st>>>(d); n_launches += 1; }
        k_compact_pos<<<grid_for(C, 8, sms), TB, 0, st>>>(d); n_launches += 1;
        d.gt_col = nullptr;
        if (d.allele_dosage && NP) { d.gt_col = dalloc<uint64_t>(NP); k_gt_columns<<<grid_for(NP, TB, sms), TB, 0, st>>>(d); n_launches += 1; }
        // ---- CSR cells of the final matrix; with host output they travel D2H on a second stream under the clustering
        d.cell_base = cell_base;
        scan(d.fr_nv, NF, d.cell_off, cell_base);
        if (NF) { if (sz.NB <= 96 * C) k_write_cells<BITS, 8><<<grid_for(NF, 32, sms), TB, 0, st>>>(d); else k_write_cells<BITS, 32><<<grid_for(NF, 8, sms), TB, 0, st>>>(d); n_launches += 1; }
        if (early_out) CK(cudaEventRecord(ln->ev_cells, st));          // the matrix part of the result is final: see copy_matrix()
        CK(cudaEventRecord(ln->ev[2], st));
        // ---- scoring
        if (nf_big) { k_read_rates<BITS><<<grid_for(NF, 8, sms), TB, 0, st>>>(d); n_launches += 1; }
        if (nf_big) { k_pair_scores<BITS><<<grid_for(NF, 8, sms), TB, 0, st>>>(d); n_launches += 1; }
        // chains above CC_MAXN reads: edge slots, lists and the maximum tree of k_cluster_sparse.  Their sizes follow from the
        // number of scored pairs per chain, known after k_read_rates: sync #2 (only when such chains exist).
        SpArrays sp{}; int sp_nmax = 0, sp_max_leaf = 0, sp_n_large = 0, sp_nmax_small = 0, sp_leaf_small = 0; unsigned sp_grid = 0;
        if (nf_sparse) {
            unsigned long long* h_pairs2 = cx->pin.get<unsigned long long>(C);
            CK(cudaMemcpyAsync(h_pairs2, d.ch_pairs2, C * 8, cudaMemcpyDeviceToHost, st));
            CK(cudaStreamSynchronize(st));
            std::vector<SpChain> chs;
            int64_t slots = 0, pool = 0, nodes = 0, leaves = 0, sups = 0;
            int firstb, lenb; range_of(CC_MAXN + 1, MAX_READS_CLUSTER, firstb, lenb);
            for (int k = 0; k < lenb; k++) {
                const int c = s_order[firstb + k];
                SpChain ch{};
                ch.chain = c; ch.n = h_nfinal[c]; ch.w_off = s_cw[c];
                const int64_t e0 = (int64_t)(h_pairs2[c] / 2) + 1;
                if (e0 > ((int64_t)1 << 30)) throw LimitFail{"a chain has more than 2^30 scored read pairs"};
                ch.slot_off = slots; ch.slot_cap = (int32_t)e0; ch.n_leaf = (int32_t)((e0 + 63) / 64); ch.n_sup = (ch.n_leaf + 63) / 64;
                ch.list_off = pool; ch.list_cap = 2 * e0 * 9 + 1024;              // the initial lists + room for the lists written by the merges
                ch.node_off = nodes; ch.leaf_off = leaves; ch.sup_off = sups;
                slots += e0; pool += ch.list_cap; nodes += ch.n; leaves += ch.n_leaf; sups += ch.n_sup;
                sp_nmax = std::max(sp_nmax, ch.n); sp_max_leaf = std::max(sp_max_leaf, ch.n_leaf);
                if (ch.n > SP_SMALL_N) sp_n_large++;                               // the list is sorted by decreasing read count
                else { sp_nmax_small = std::max(sp_nmax_small, ch.n); sp_leaf_small = std::max(sp_leaf_small, ch.n_leaf); }
                chs.push_back(ch);
            }
            if (sp_smem_bytes(sp_nmax, sp_max_leaf) > cx->smem_optin) throw LimitFail{"a chain's cluster-editing state exceeds the shared memory of a block"};
            sp.n_chains = (int)chs.size(); sp.n_nodes = nodes; sp.n_slot_cap = slots; sp.n_leaves = leaves; sp.n_sups = sups;
            sp.fl_slot = dalloc<uint32_t>(slots); sp.fl_old = dalloc<int32_t>(slots); sp.supq = dalloc<uint32_t>(sups); sp.leafq = dalloc<uint32_t>(leaves);
            sp.chains = up_pinned(chs.data(), (int64_t)chs.size());
            sp.key = dalloc<uint32_t>(slots); sp.flag = dalloc<uint8_t>(slots); sp.F = (long long*)dalloc<int64_t>(slots); sp.P = (long long*)dalloc<int64_t>(slots);
            sp.pool = dalloc<uint32_t>(pool);
            sp.lptr = (long long*)dalloc<int64_t>(nodes); sp.llen = dalloc<uint32_t>(nodes); sp.sa = dalloc<uint32_t>(nodes); sp.sb = dalloc<uint32_t>(nodes); sp.up = dalloc<uint32_t>(nodes);
            sp.wa = dalloc<int32_t>(nodes); sp.wb = dalloc<int32_t>(nodes); sp.nw = dalloc<int32_t>(nodes);
            sp.frF = (long long*)dalloc<int64_t>(nodes); sp.frP = (long long*)dalloc<int64_t>(nodes);
            sp.leaf = (SpBest*)cx->dev.alloc((size_t)std::max<int64_t>(leaves, 1) * sizeof(SpBest)); sp.sup = (SpBest*)cx->dev.alloc((size_t)std::max<int64_t>(sups, 1) * sizeof(SpBest));
            sp.bump = (long long*)dalloc<int64_t>((int64_t)chs.size()); sp.n_slots = dalloc<int32_t>((int64_t)chs.size());
            sp_grid = (unsigned)grid_for(nodes, 8, sms);
            k_sp_degrees<<<sp_grid, TB, 0, st>>>(d, sp); k_sp_scan<<<(unsigned)chs.size(), 1024, 0, st>>>(sp);
            k_sp_fill<<<sp_grid, TB, 0, st>>>(d, sp); k_sp_init_costs<<<(unsigned)grid_for(slots, 8, sms), TB, 0, st>>>(d, sp);
            k_sp_leaves<<<(unsigned)grid_for(leaves, 8, sms), TB, 0, st>>>(sp); k_sp_sups<<<(unsigned)grid_for(sups, 8, sms), TB, 0, st>>>(sp);
            n_launches += 6;
            CK(cudaGetLastError());
        }
        // chains up to CC_MAXN reads: scoring out of shared memory, 4 B per pair to HBM (every chain of BASELINE config 2).
        // The size classes run side by side on the side streams: one class alone leaves issue slots idle (barrier waits).
        CK(cudaEventRecord(ln->ev_fork, st));
        for (auto& t : cx->side) CK(cudaStreamWaitEvent(t, ln->ev_fork, 0));
        for (int k = N_SCORE - 1, q = 0; k >= 0; k--) {
            int first, len; range_of(k ? kScore[k - 1].nmax + 1 : 1, kScore[k].nmax, first, len);
            if (!len) continue;
            const int nt = kScore[k].nt;
            const size_t smem = cs_smem_bytes(kScore[k].nmax, kScore[k].nt);
            const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(std::min<size_t>(16, 2048 / nt), (228 * 1024) / (smem + 1024)));
            const unsigned grid = (unsigned)std::min<int64_t>(len, (int64_t)sms * per_sm);
            score_launch<BITS>(nt, kScore[k].kpl, grid, smem, cx->side[q++ & 7], d, dv_order + first, len, kScore[k].nmax, counters + 8 + k); n_launches += 1;
        }
        for (int i = 0; i < 8; i++) { CK(cudaEventRecord(ln->ev_join[i], cx->side[i])); CK(cudaStreamWaitEvent(st, ln->ev_join[i], 0)); }
        CK(cudaEventRecord(ln->ev[3], st));
        // ---- cluster editing out of shared memory
        // the size classes run on four side streams so that the tail of one class overlaps the bulk of the next
        CK(cudaEventRecord(ln->ev_fork, st));
        for (auto& t : cx->side) CK(cudaStreamWaitEvent(t, ln->ev_fork, 0));
        for (int k = N_CLUSTER - 1, q = 0; k >= 0; k--) {
            int first, len; range_of(k ? kCluster[k - 1].nmax + 1 : 1, kCluster[k].nmax, first, len);
            if (!len) continue;
            const int nt = kCluster[k].nt;
            const size_t smem = cc_smem_bytes(kCluster[k].nmax, nt);
            const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(std::min<size_t>(cc_min_blocks(nt, kCluster[k].per), 2048 / nt), (228 * 1024) / (smem + 1024)));
            const unsigned grid = (unsigned)std::min<int64_t>(len, (int64_t)sms * per_sm);
            int32_t* scratch = dalloc<int32_t>((int64_t)grid * nt * kCluster[k].per * 3);     // slot-packing areas, one per warp
            cluster_launch(nt, kCluster[k].per, grid, smem, cx->side[q++ & 7], d, dv_order + first, len, kCluster[k].nmax, counters + 8 + N_SCORE + k, scratch); n_launches += 1;
        }
        // ---- cluster editing of the chains above CC_MAXN reads, on two of the side streams (next to the shared-memory classes)
        if (sp.n_chains) {
            // the few long chains in blocks of 1024 threads, the many short ones (<= 1024 reads) 256 threads each, several per SM:
            // a greedy step is a chain of dependent memory latencies, which only other chains can hide
            if (sp_n_large) {
                k_cluster_sparse<SP_THREADS><<<(unsigned)std::min<int64_t>(sp_n_large, sms), SP_THREADS, sp_smem_bytes(sp_nmax, sp_max_leaf), cx->side[7]>>>(d, sp, 0, sp_n_large, sp_nmax, sp_max_leaf, counters + 2);
                n_launches += 1;
            }
            if (sp.n_chains > sp_n_large) {
                const size_t sm_small = sp_smem_bytes(sp_nmax_small, sp_leaf_small);
                const int per_sm = (int)std::max<size_t>(1, std::min<size_t>(8, (200 * 1024) / (sm_small + 1024)));
                k_cluster_sparse<SP_THREADS_SMALL><<<(unsigned)std::min<int64_t>(sp.n_chains - sp_n_large, (int64_t)sms * per_sm), SP_THREADS_SMALL, sm_small, cx->side[6]>>>(d, sp, sp_n_large, sp.n_chains, sp_nmax_small, sp_leaf_small, counters + 3);
                n_launches += 1;
            }
        }
        for (int i = 0; i < 8; i++) { CK(cudaEventRecord(ln->ev_join[i], cx->side[i])); CK(cudaStreamWaitEvent(st, ln->ev_join[i], 0)); }
        CK(cudaEventRecord(ln->ev[4], st));
        // ---- coverage / consensus, threading
        if (NP && BITS == 2) { k_consensus_chain<<<grid_for(C, 4, sms), 128, 0, st>>>(d); n_launches += 1; }      // chains with <= 16 clusters
        if (NP) {                                          // the rest: 16 lanes per position while the depth (reads per chain) is small
            if (NF <= 96 * C) k_consensus<BITS, 16><<<grid_for(NP, 8, sms), 128, 0, st>>>(d); else k_consensus<BITS, 32><<<grid_for(NP, 4, sms), 128, 0, st>>>(d);
            n_launches += 1;
        }
        CK(cudaEventRecord(ln->ev[5], st));
        if (NP && in->ploidy == 2) { k_thread2<<<(unsigned)std::min<int64_t>((C + 7) / 8, (int64_t)sms * 8), 256, 0, st>>>(d, counters + 1); n_launches += 1; }
        else if (NP && in->ploidy <= 4) { k_thread<<<std::min<int64_t>(C, (int64_t)sms * 8), DP_THREADS, 21 * (size_t)S_max + 64, st>>>(d, counters + 1); n_launches += 1; }
        else if (NP) {
            const unsigned grid = (unsigned)std::min<int64_t>(C, (int64_t)sms * 4);
            if (d.gt_col) k_thread_canon<true><<<grid, CN_THREADS, 64 * 1024, st>>>(d, cx->canon, counters + 1);
            else k_thread_canon<false><<<grid, CN_THREADS, 64 * 1024, st>>>(d, cx->canon, counters + 1);
            n_launches += 1;
        }
        CK(cudaEventRecord(ln->ev[6], st));
        CK(cudaGetLastError());
    }

    void run_phase2() { if (d.bits == 2) run_bits<2>(); else run_bits<4>(); }
    void run() { run_phase1_enqueue(); run_phase1_finish(); run_phase2(); }

    void collect_times() {
        float t;
        CK(cudaEventElapsedTime(&t, ln->ev[0], ln->ev[1])); ms[0] = t;
        CK(cudaEventElapsedTime(&t, ln->ev[1], ln->ev[2])); ms[1] = t;
        CK(cudaEventElapsedTime(&t, ln->ev[2], ln->ev[3])); ms[2] = t;
        CK(cudaEventElapsedTime(&t, ln->ev[3], ln->ev[4])); ms[3] = t;
        CK(cudaEventElapsedTime(&t, ln->ev[4], ln->ev[5])); ms[4] = t;
        CK(cudaEventElapsedTime(&t, ln->ev[5], ln->ev[6])); ms[5] = t;
        CK(cudaEventElapsedTime(&t, ln->ev[0], ln->ev[6])); ms[6] = t;
    }

    // where this pipeline's results go inside the arrays of ahs_batch_out (a chunk writes a slice)
    struct Slices {
        int32_t *status, *read_id, *read_mapq, *read_cluster, *cell_pos, *n_clusters, *pos, *path, *maxpos;
        int64_t* cell_off; uint8_t *cell_allele, *hap_allele; double* dp_cost; bool first_chunk;
    };
    template <class T> void cp(T* h, const T* dptr, int64_t n, cudaStream_t st) {
        if (n > 0) CK(cudaMemcpyAsync(h, dptr, n * sizeof(T), cudaMemcpyDeviceToHost, st));
    }
    // the allele matrix and the read order are final after k_write_cells: they travel on the second stream while the
    // clustering runs (early_out), or with the rest
    void copy_matrix(const Slices& o, cudaStream_t st) {
        const int64_t NF = d.NF, NP = d.NP;
        cp(o.read_id, d.fr_id, NF, st); cp(o.read_mapq, d.fr_mapq, NF, st);
        if (o.first_chunk) cp(o.cell_off, d.cell_off, NF + 1, st); else cp(o.cell_off + 1, d.cell_off + 1, NF, st);   // entry 0 = the previous chunk's last
        cp(o.cell_pos, d.cell_pos, h_tot_cells, st); cp(o.cell_allele, d.cell_allele, h_tot_cells, st); cp(o.pos, d.pos, NP, st);
    }
    void copy_rest(const Slices& o, int64_t* h_pairs) {
        const int64_t C = sz.C, NF = d.NF, NP = d.NP; const int p = in->ploidy;
        cudaStream_t st = ln->stream;
        cp(o.status, d.ch_status, C, st); cp(o.read_cluster, d.fr_cluster, NF, st); cp(o.n_clusters, d.ch_nclusters, C, st);
        cp(o.path, d.path, NP * p, st); cp(o.hap_allele, d.hap_allele, NP * p, st); cp(o.dp_cost, d.dp_cost, C, st); cp(o.maxpos, d.ch_maxpos, C, st);
        CK(cudaMemcpyAsync(h_pairs, d.tot_pairs, 8, cudaMemcpyDeviceToHost, st));
    }
};

static int guarded(const char* what, const std::function<void()>& fn) {
    try { fn(); g_err[0] = 0; return AHS_OK; }
    catch (const CudaFail& f) { set_err("%s: CUDA error %d (%s) at %s, line %d", what, (int)f.e, cudaGetErrorString(f.e), f.what, f.line); cudaGetLastError(); return AHS_ERR_CUDA; }
    catch (const LimitFail& f) { set_err("%s: limit exceeded: %s", what, f.msg.c_str()); return AHS_ERR_LIMIT; }
    catch (const ArgFail& f) { set_err("%s: bad argument: %s", what, f.msg.c_str()); return AHS_ERR_ARG; }
    catch (const PassThrough& f) { set_err("%s: %s", what, f.msg.c_str()); return f.rc; }
    catch (const std::exception& e) { set_err("%s: %s", what, e.what()); return AHS_ERR_INTERNAL; }
}

static void fill_empty_out(ahs_batch_out* out, Ctx* cx, int ploidy) {
    memset(out, 0, sizeof(*out));
    out->ploidy = ploidy;
    out->read_off = cx->outp.get<int64_t>(1); out->read_off[0] = 0;
    out->pos_off = cx->outp.get<int64_t>(1); out->pos_off[0] = 0;
    out->cell_off = cx->outp.get<int64_t>(1); out->cell_off[0] = 0;
}

struct HostTrace {       // AHS_TRACE=1: wall-clock of the host-side steps of one call, on stderr
    bool on; std::chrono::steady_clock::time_point t0; std::string line;
    HostTrace() : on(getenv("AHS_TRACE") != nullptr), t0(std::chrono::steady_clock::now()) {}
    void mark(const char* what) {
        if (!on) return;
        const auto t1 = std::chrono::steady_clock::now();
        char buf[96]; snprintf(buf, sizeof buf, " %s=%.2fms", what, std::chrono::duration<double, std::milli>(t1 - t0).count());
        line += buf; t0 = t1;
    }
    void note(const char* what, double v) { if (on) { char buf[96]; snprintf(buf, sizeof buf, " %s=%.1f", what, v); line += buf; } }
    ~HostTrace() { if (on) fprintf(stderr, "[ahs trace]%s\n", line.c_str()); }
};

// a range of consecutive chains as a batch of its own: the big arrays are slices of the caller's (their offsets are
// rebased on the device after the upload), the three per-chain offset arrays are rebased here
struct Range { int64_t c0, c1; };

struct ChainView {
    // the three rebased offset arrays live in page-locked staging: an async copy from pageable memory would first drain the
    // stream it is enqueued on (and with it the upload of the range before)
    ahs_batch_in v; int64_t *bubble_off = nullptr, *read_off = nullptr, *entry_off = nullptr;
    const uint8_t* dosage = nullptr;                    // the caller's allele dosages from the range's first allele on, like anode_off
    void make(const ahs_batch_in* in, const uint8_t* in_dosage, int64_t c0, int64_t c1, Pool& pin) {
        const int64_t C = in->n_chains, NB = in->bubble_off[C], NE = in->entry_off[C];
        const int64_t n = c1 - c0, b0 = in->bubble_off[c0], e0 = in->entry_off[c0];
        // the interior offsets dereferenced below are checked here; everything else is validated on the device
        const int64_t NA = in->allele_off[NB] , a0 = in->allele_off[b0], a1 = in->allele_off[in->bubble_off[c1]];
        if (a0 < 0 || a1 < a0 || a1 > NA) throw ArgFail{"allele_off / anode_off / enode_off not monotone"};
        const int64_t NAN_ = in->anode_off[NA], an0 = in->anode_off[a0], an1 = in->anode_off[a1];
        const int64_t NEN = in->enode_off[NE], en0 = in->enode_off[e0], en1 = in->enode_off[in->entry_off[c1]];
        if (an0 < 0 || an1 < an0 || an1 > NAN_ || en0 < 0 || en1 < en0 || en1 > NEN) throw ArgFail{"allele_off / anode_off / enode_off not monotone"};
        bubble_off = pin.get<int64_t>((size_t)n + 1); read_off = pin.get<int64_t>((size_t)n + 1); entry_off = pin.get<int64_t>((size_t)n + 1);
        for (int64_t c = 0; c <= n; c++) { bubble_off[c] = in->bubble_off[c0 + c] - b0; read_off[c] = in->read_off[c0 + c] - in->read_off[c0]; entry_off[c] = in->entry_off[c0 + c] - e0; }
        v = *in;
        v.n_chains = (int32_t)n; v.chain_id = in->chain_id ? in->chain_id + c0 : nullptr;
        v.bubble_off = bubble_off; v.read_off = read_off; v.entry_off = entry_off;
        v.allele_off = in->allele_off + b0; v.anode_off = in->anode_off + a0; v.anode = in->anode + an0;
        dosage = in_dosage ? in_dosage + a0 : nullptr;
        v.stage_a_order = in->stage_a_order ? in->stage_a_order + b0 : nullptr;
        v.enode_off = in->enode_off + e0; v.enode = in->enode + en0;
        v.entry_read = in->entry_read + e0; v.entry_identity = in->entry_identity + e0;
    }
};

// the output arrays of a call: allocated once the sizes of every range are known, from the page-locked result pool of
// the call's first device (portable: every device of the call copies its ranges straight into them)
static void alloc_out(ahs_batch_out* out, Ctx* cx, int64_t C, int p, int64_t NFt, int64_t NPt, int64_t cells) {
    memset(out, 0, sizeof(*out));
    out->n_chains = (int32_t)C; out->ploidy = p;
    out->status = cx->outp.get<int32_t>(C); out->n_clusters = cx->outp.get<int32_t>(C); out->dp_cost = cx->outp.get<double>(C); out->maxpos = cx->outp.get<int32_t>(C);
    out->read_off = cx->outp.get<int64_t>(C + 1); out->pos_off = cx->outp.get<int64_t>(C + 1);
    out->read_id = cx->outp.get<int32_t>(std::max<int64_t>(NFt, 1)); out->read_mapq = cx->outp.get<int32_t>(std::max<int64_t>(NFt, 1));
    out->read_cluster = cx->outp.get<int32_t>(std::max<int64_t>(NFt, 1)); out->cell_off = cx->outp.get<int64_t>(NFt + 1);
    out->cell_pos = cx->outp.get<int32_t>(std::max<int64_t>(cells, 1)); out->cell_allele = cx->outp.get<uint8_t>(std::max<int64_t>(cells, 1));
    out->pos = cx->outp.get<int32_t>(std::max<int64_t>(NPt, 1)); out->path = cx->outp.get<int32_t>(std::max<int64_t>(NPt * p, 1));
    out->hap_allele = cx->outp.get<uint8_t>(std::max<int64_t>(NPt * p, 1));
    out->read_off[0] = 0; out->pos_off[0] = 0; out->cell_off[0] = 0;
}

// Everything one device does for one call: its ranges of chains run as pipelines on the context's lanes (range k+1
// uploads and projects under the clustering of range k, so that most of the H2D time is hidden), then — once the
// caller has placed every range in the output arrays — the results are copied straight into their slices.
struct DeviceJob {
    Ctx* cx = nullptr; int device = -1; const ahs_batch_in* in = nullptr; const uint8_t* dosage = nullptr;
    std::vector<Range> ranges;
    std::vector<ChainView> views; std::vector<Pipeline> pls; std::vector<Sizes> szs;
    std::unique_lock<std::mutex> lock;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
    float acc[7] = {0}, h2d = 0, d2h = 0;
    int iters = 0; int64_t* h_pairs = nullptr;
    HostTrace tr;

    void begin(int dev, const ahs_batch_in* in_, const uint8_t* dosage_) {
        device = dev; in = in_; dosage = dosage_;
        cx = get_ctx(device);
        lock = std::unique_lock<std::mutex>(cx->mu);
        tr.mark("context");
        CK(cudaSetDevice(device));
        if (cx->out_busy) throw ArgFail{"previous ahs_batch_out of this device was not released with ahs_free_out"};
        CK(cudaDeviceSynchronize());                          // nothing of a failed earlier call is in flight
        cx->dev.reset(); cx->outp.reset(); cx->pin.reset();
    }

    // phase 1 (ends with sync #1 per range) and phase 2 of every range, enqueued
    void enqueue(int warmup, int iters_) {
        iters = iters_;
        const int n = (int)ranges.size();
        views.resize(n); pls.resize(n); szs.resize(n);
        e0 = cx->lanes[0].ev[7]; e1 = cx->lanes[0].ev[8];
        CK(cudaSetDevice(device));
        CK(cudaEventRecord(e0, cx->lanes[0].stream));
        bool first = true; Lane* last_up = nullptr;
        // range k+1 is prepared and its upload enqueued once phase 2 of range k is enqueued: it travels under the clustering of
        // range k.  AHS_UPLOAD_AHEAD=1 does it one step earlier, under phase 1 of range k (the uploads then follow each other
        // on the copy engine without gaps); measured 1 ms slower end to end on one device (cfg2: 42.6 vs 41.6 ms), kept as a knob.
        auto prepare = [&](int k) {
            Pipeline& pl = pls[k];
            pl.cx = cx; pl.ln = &cx->lanes[k % N_LANES]; pl.early_out = iters == 0;
            if (n == 1 && ranges[0].c0 == 0 && ranges[0].c1 == in->n_chains) { pl.in = in; pl.dosage = dosage; pl.sz = validate(in); }
            else { views[k].make(in, dosage, ranges[k].c0, ranges[k].c1, cx->pin); pl.in = &views[k].v; pl.dosage = views[k].dosage; pl.sz = validate(pl.in, true); }
            szs[k] = pl.sz;
            if (pl.sz.C == 0) return;
            pl.upload(last_up);
            last_up = pl.ln;
            if (first) { CK(cudaEventRecord(e1, pl.ln->stream)); tr.mark("upload_enqueue"); first = false; }
            pl.alloc_phase1();
        };
        const bool ahead = getenv("AHS_UPLOAD_AHEAD") && atoi(getenv("AHS_UPLOAD_AHEAD")) != 0;
        if (n > 0) prepare(0);
        for (int k = 0; k < n; k++) {
            Pipeline& pl = pls[k];
            if (iters > 0) {
                if (pl.sz.C == 0) continue;
                // the device pool is bump-allocated: remember the mark so that resident iterations reuse phase-2 space
                std::vector<size_t> mark; for (auto& c : cx->dev.chunks) mark.push_back(c.used);
                for (int it = 0; it < warmup + iters; it++) {
                    for (size_t i = 0; i < cx->dev.chunks.size(); i++) cx->dev.chunks[i].used = i < mark.size() ? mark[i] : 0;
                    pl.run();
                    CK(cudaStreamSynchronize(pl.ln->stream));
                    pl.collect_times();
                    if (it >= warmup) for (int i = 0; i < 7; i++) acc[i] += pl.ms[i];
                }
                if (k + 1 < n) prepare(k + 1);
                continue;
            }
            if (pl.sz.C) { pl.run_phase1_enqueue(); tr.mark("phase1_enqueue"); }
            if (ahead && k + 1 < n) { prepare(k + 1); tr.mark("prepare"); }            // host work and upload of the next range under this range's phase 1
            if (pl.sz.C) { pl.run_phase1_finish(); tr.mark("sync1"); pl.run_phase2(); tr.mark("phase2_enqueue"); }
            if (!ahead && k + 1 < n) { prepare(k + 1); tr.mark("prepare"); }
        }
        if (first) CK(cudaEventRecord(e1, cx->lanes[0].stream));
    }

    // copies of every range into its slices of `out`; f_base / q_base / cell_base: final reads, positions and cells of
    // the ranges that precede range k in chain order (over all devices of the call)
    void copy_out(ahs_batch_out* out, const int64_t* f_base, const int64_t* q_base, const int64_t* cell_base) {
        const int n = (int)ranges.size(); const int p = in->ploidy;
        CK(cudaSetDevice(device));
        h_pairs = cx->pin.get<int64_t>(std::max(n, 1));
        CK(cudaEventSynchronize(e1)); CK(cudaEventElapsedTime(&h2d, e0, e1));
        cudaEvent_t d0 = cx->lanes[0].ev[7];
        CK(cudaEventRecord(d0, cx->lanes[0].stream2));
        for (int k = 0; k < n; k++) {
            h_pairs[k] = 0;
            if (szs[k].C == 0) continue;
            Pipeline& pl = pls[k];
            const int64_t c0 = ranges[k].c0, f = f_base[k], q = q_base[k], cells = cell_base[k];
            Pipeline::Slices sl{out->status + c0, out->read_id + f, out->read_mapq + f, out->read_cluster + f, out->cell_pos + cells, out->n_clusters + c0,
                                out->pos + q, out->path + q * p, out->maxpos + c0, out->cell_off + f, out->cell_allele + cells, out->hap_allele + q * p,
                                out->dp_cost + c0, false};
            for (int64_t c = 0; c < szs[k].C; c++) { out->read_off[c0 + c + 1] = f + pl.h_frow_off[c + 1]; out->pos_off[c0 + c + 1] = q + pl.h_pos_off[c + 1]; }
            cudaStream_t ms = pl.early_out ? pl.ln->stream2 : pl.ln->stream;
            if (pl.early_out) CK(cudaStreamWaitEvent(ms, pl.ln->ev_cells, 0));
            if (cells && pl.d.NF) { k_rebase<<<grid_for(pl.d.NF + 1, 256, cx->sms), 256, 0, ms>>>(pl.d.cell_off, pl.d.NF + 1, -cells); CK(cudaGetLastError()); }
            pl.copy_matrix(sl, ms);
            pl.copy_rest(sl, h_pairs + k);
        }
        tr.mark("copies_enqueue");
        for (int k = 0; k < std::min(n, N_LANES); k++) { CK(cudaStreamSynchronize(cx->lanes[k].stream2)); CK(cudaStreamSynchronize(cx->lanes[k].stream)); }
        tr.mark("run_sync");
        {
            auto mb = [](const Pool& p, bool used) { double t = 0; for (auto& c : p.chunks) t += (double)(used ? c.used : c.cap); return t / 1048576.0; };
            tr.note("dev_used_mb", mb(cx->dev, true)); tr.note("dev_cap_mb", mb(cx->dev, false));
            tr.note("pin_used_mb", mb(cx->pin, true)); tr.note("out_used_mb", mb(cx->outp, true));
        }
        CK(cudaEventRecord(e1, cx->lanes[0].stream)); CK(cudaEventSynchronize(e1));
        CK(cudaEventElapsedTime(&d2h, d0, e1));
    }

    // stage times of this device: summed over its ranges (resident mode: averaged over the timed iterations)
    void times(float* ms7, int& launches) {
        const int n = (int)ranges.size();
        for (int i = 0; i < 7; i++) ms7[i] = 0;
        launches = 0;
        if (iters > 0) { for (int i = 0; i < 7; i++) ms7[i] = acc[i] / iters; for (auto& pl : pls) launches += pl.n_launches; return; }
        int firstk = -1, last = -1;
        for (int k = 0; k < n; k++) if (szs[k].C) {
            if (n <= N_LANES) { pls[k].collect_times(); for (int i = 0; i < 6; i++) ms7[i] += pls[k].ms[i]; }      // a lane's events are re-recorded by a later range
            launches += pls[k].n_launches;
            if (firstk < 0) firstk = k; last = k;
        }
        if (firstk >= 0 && n <= N_LANES) { float t = 0; CK(cudaEventElapsedTime(&t, pls[firstk].ln->ev[0], pls[last].ln->ev[6])); ms7[6] = t; }      // first kernel -> last kernel
        if (getenv("AHS_TRACE") && n <= N_LANES)          // device timeline of the ranges, ms after the call's first event
            for (int k = 0; k < n; k++) if (szs[k].C) {
                auto at = [&](cudaEvent_t e) { float t = 0; CK(cudaEventElapsedTime(&t, e0, e)); return t; };
                Lane* l = pls[k].ln;
                fprintf(stderr, "[ahs timeline] dev %d range %d chains %lld: uploaded %.2f | phase1 start %.2f front %.2f rows+sync1 %.2f score %.2f cluster %.2f consensus %.2f thread %.2f\n",
                        device, k, (long long)szs[k].C, at(l->ev_up), at(l->ev[0]), at(l->ev[1]), at(l->ev[2]), at(l->ev[3]), at(l->ev[4]), at(l->ev[5]), at(l->ev[6]));
            }
    }
};

// Ranges of the chains [cb, ce) of a call on one device; iters > 0 = resident timing mode.  A call with host output
// (iters == 0) and a large share runs as three ranges of chains (12 % / 41 % / 47 % of the alignment nodes, the bulk of the
// upload): range k+1 uploads under the clustering of range k.
static std::vector<Range> ranges_of_share(const ahs_batch_in* in, const Sizes& sz, int64_t cb, int64_t ce, int iters) {
    const int64_t C = ce - cb;
    auto en_at = [&](int64_t c) -> int64_t {                 // alignment nodes before chain c
        const int64_t e = in->entry_off[c];
        if (e < 0 || e > sz.NE) throw ArgFail{"entry_off out of range"};
        return in->enode_off[e];
    };
    const int64_t en0 = en_at(cb), NEN = en_at(ce) - en0;
    int n_chunks = 1;
    if (iters == 0 && C >= 4096 && NEN >= (int64_t)16 << 20) {
        n_chunks = 3;
        // ranges pay (tails of the cluster-editing launches, three host syncs; the big chains of different ranges run one after
        // the other) where there is an upload worth hiding: not when the estimated device time (ahs_chain_cost, ~7.4 us a unit
        // on one B200) dwarfs the transfer (~55 GB/s), nor when one long chain's sequential merges (>= 30 us each) do
        double units = 0; int64_t max_entries = 0;
        for (int64_t c = cb; c < ce; c++) {
            const int64_t e0 = in->entry_off[c], e1 = in->entry_off[c + 1];
            if (e0 < 0 || e1 < e0 || e1 > sz.NE) throw ArgFail{"entry_off out of range"};
            units += ahs_chain_cost(in->bubble_off[c + 1] - in->bubble_off[c], e1 - e0, in->enode_off[e1] - in->enode_off[e0], in->ploidy);
            max_entries = std::max(max_entries, e1 - e0);
        }
        const double upload_ms = (double)NEN * 4.0 / 55e6, nf_max = 0.7 * (double)max_entries;
        if (upload_ms < 0.03 * units * 7.4e-3 || (nf_max > 160.0 && upload_ms < 0.1 * nf_max * 0.03)) n_chunks = 1;
        if (const char* e = getenv("AHS_CHUNKS")) n_chunks = std::max(1, std::min(N_LANES, atoi(e)));       // tuning / debugging
    }
    std::vector<int64_t> cut(n_chunks + 1, cb); cut[n_chunks] = ce;
    // the first chunk is the smallest: nothing runs under its upload, and it only has to cover the next chunk's
    std::vector<double> frac(n_chunks + 1, 1.0);
    for (int k = 0; k <= n_chunks; k++) frac[k] = (double)k / n_chunks;
    if (n_chunks == 3) { frac[1] = 0.12; frac[2] = 0.53; }
    if (const char* e = getenv("AHS_CUTS")) {                // tuning / debugging: "0.2,0.6"
        const char* q = e;
        for (int k = 1; k < n_chunks && *q; k++) { frac[k] = std::min(1.0, std::max(frac[k - 1], atof(q))); while (*q && *q != ',') q++; if (*q == ',') q++; }
    }
    for (int k = 1; k < n_chunks; k++) {
        const int64_t target = en0 + (int64_t)((double)NEN * frac[k]);
        int64_t lo = cut[k - 1], hi = ce;                 // first chain whose entries start at or after the target
        while (lo < hi) { const int64_t mid = (lo + hi) / 2; if (en_at(mid) >= target) hi = mid; else lo = mid + 1; }
        cut[k] = lo;
    }
    std::vector<Range> r;
    for (int k = 0; k < n_chunks; k++) r.push_back(Range{cut[k], cut[k + 1]});
    return r;
}

// Multi-device plan (SURVEY §8e): every device gets ONE contiguous share of the chains, cut so that the largest estimated
// share cost (ahs_chain_cost) is as small as contiguous cuts allow (binary search on the bound, greedy packing on prefix sums),
// and runs it like a single-device call (ranges_of_share).  The chains arrive largest first (size_sorting,
// polyassembly.cpp:135-140): the long chains of a share sit in one range and cluster side by side on different SMs.  (The first
// version dealt heavy chains one by one, largest first onto the least loaded device: balanced on paper, but a device ran its
// single-chain ranges one after the other — 1.49 s on two devices against 0.85 s on one for the Zipf-skewed batch.)
// The shares are ranges of the caller's arrays: uploaded and downloaded in place, nothing is re-packed on the host.
static std::vector<std::vector<Range>> plan_devices(const ahs_batch_in* in, const Sizes& sz, int G, std::vector<double>* load_out) {
    const int64_t C = sz.C; const int p = in->ploidy;
    std::vector<double> pre(C + 1, 0.0);
    for (int64_t c = 0; c < C; c++) {
        const int64_t e0 = in->entry_off[c], e1 = in->entry_off[c + 1];
        if (e0 < 0 || e1 < e0 || e1 > sz.NE) throw ArgFail{"entry_off out of range"};
        const double k = ahs_chain_cost(in->bubble_off[c + 1] - in->bubble_off[c], e1 - e0, in->enode_off[e1] - in->enode_off[e0], p);
        pre[c + 1] = pre[c] + k;
    }
    const std::vector<int64_t> cuts = balanced_contiguous_cuts(pre, G);                  // host_plan.hpp
    std::vector<std::vector<Range>> plan(G); std::vector<double> load(G, 0.0);
    for (int g = 0; g < G; g++) {
        if (cuts[g + 1] > cuts[g]) plan[g] = ranges_of_share(in, sz, cuts[g], cuts[g + 1], 0);
        load[g] = pre[cuts[g + 1]] - pre[cuts[g]];
    }
    if (load_out) *load_out = load;
    return plan;
}

// small reusable barrier for the device threads of one call
struct ThreadBarrier {
    std::mutex m; std::condition_variable cv; int n, waiting = 0, gen = 0;
    explicit ThreadBarrier(int n_) : n(n_) {}
    void arrive() { std::unique_lock<std::mutex> l(m); const int g = gen; if (++waiting == n) { waiting = 0; gen++; cv.notify_all(); } else cv.wait(l, [&] { return gen != g; }); }
};

// one batch on the given devices.  G == 1: the whole batch on that device.  G > 1: plan_devices(); one host thread per
// device; no inter-GPU traffic; every device writes its ranges straight into the (portable, page-locked) output arrays.
static void phase_on_devices(const ahs_batch_in* in, const uint8_t* dosage, ahs_batch_out* out, const int* devs, int G, int warmup, int iters) {
    if (!out) throw ArgFail{"null output"};
    if (!devs || G < 1) throw ArgFail{"no devices"};
    for (int g = 0; g < G; g++) for (int h = 0; h < g; h++) if (devs[g] == devs[h]) throw ArgFail{"ahs_phase_batch_multi: a device id is listed twice"};
    struct RestoreDevice {          // the caller's current device is the caller's business: put it back on every way out
        int dev = -1;
        RestoreDevice() { if (cudaGetDevice(&dev) != cudaSuccess) { dev = -1; cudaGetLastError(); } }
        ~RestoreDevice() { if (dev >= 0) cudaSetDevice(dev); }
    } restore_device;
    Sizes sz = validate(in);
    const int64_t C = sz.C; const int p = in->ploidy;
    std::vector<DeviceJob> jobs(G);
    if (C == 0) {
        jobs[0].begin(devs[0], in, dosage);
        fill_empty_out(out, jobs[0].cx, p); jobs[0].cx->out_busy = true;
        jobs[0].lock.unlock();
        return;
    }
    std::vector<std::vector<Range>> plan;
    std::vector<double> load;
    if (G == 1) plan.push_back(ranges_of_share(in, sz, 0, C, iters)); else plan = plan_devices(in, sz, G, &load);
    // every range of the call, in chain order: (device, index within the device)
    struct Place { int64_t c0; int g, k; };
    std::vector<Place> places;
    for (int g = 0; g < G; g++) for (int k = 0; k < (int)plan[g].size(); k++) places.push_back(Place{plan[g][k].c0, g, k});
    std::sort(places.begin(), places.end(), [](const Place& a, const Place& b) { return a.c0 < b.c0; });
    std::vector<std::vector<int64_t>> f_base(G), q_base(G), cell_base(G);
    for (int g = 0; g < G; g++) { f_base[g].assign(plan[g].size(), 0); q_base[g] = f_base[g]; cell_base[g] = f_base[g]; }
    std::vector<std::string> errs(G); std::vector<int> rcs(G, AHS_OK);
    ThreadBarrier bar(G);
    int64_t NFt = 0, NPt = 0, tot_cells = 0;
    auto any_failed = [&]() { for (int g = 0; g < G; g++) if (rcs[g] != AHS_OK) return true; return false; };
    auto body = [&](int g) {
        DeviceJob& job = jobs[g];
        rcs[g] = guarded("device", [&]() { job.begin(devs[g], in, dosage); job.ranges = plan[g]; job.enqueue(warmup, iters); });
        if (rcs[g] != AHS_OK) errs[g] = g_err;
        bar.arrive();
        if (g == 0 && !any_failed()) {
            rcs[0] = guarded("output", [&]() {
                for (auto& pc : places) {
                    Pipeline& pl = jobs[pc.g].pls[pc.k];
                    f_base[pc.g][pc.k] = NFt; q_base[pc.g][pc.k] = NPt; cell_base[pc.g][pc.k] = tot_cells;
                    if (jobs[pc.g].szs[pc.k].C == 0) continue;
                    NFt += pl.d.NF; NPt += pl.d.NP; tot_cells += pl.h_tot_cells;
                }
                alloc_out(out, jobs[0].cx, C, p, NFt, NPt, tot_cells);
                jobs[0].cx->out_busy = true;                       // under the context's lock; taken back below if the call fails
            });
            if (rcs[0] != AHS_OK) errs[0] = g_err;
        }
        bar.arrive();
        if (!any_failed()) {
            rcs[g] = guarded("device", [&]() { job.copy_out(out, f_base[g].data(), q_base[g].data(), cell_base[g].data()); });
            if (rcs[g] != AHS_OK) errs[g] = g_err;
        } else if (job.cx) { cudaSetDevice(devs[g]); cudaDeviceSynchronize(); cudaGetLastError(); }
        if (job.lock.owns_lock()) job.lock.unlock();            // by the thread that took it
    };
    if (G == 1) body(0);
    else { std::vector<std::thread> th; for (int g = 0; g < G; g++) th.emplace_back(body, g); for (auto& t : th) t.join(); }
    for (int g = 0; g < G; g++) if (rcs[g] != AHS_OK) {
        if (jobs[0].cx) { std::lock_guard<std::mutex> l(jobs[0].cx->mu); jobs[0].cx->out_busy = false; jobs[0].cx->outp.reset(); }
        const std::string msg = G > 1 ? "device " + std::to_string(devs[g]) + ": " + errs[g] : errs[g];
        if (rcs[g] == AHS_ERR_ARG) throw ArgFail{msg};
        if (rcs[g] == AHS_ERR_LIMIT) throw LimitFail{msg};
        if (rcs[g] == AHS_ERR_CUDA) throw PassThrough{AHS_ERR_CUDA, msg};
        throw std::runtime_error(msg);
    }
    if (out->cell_off[NFt] != tot_cells) throw std::runtime_error("cell count mismatch");
    out->n_cells = tot_cells;
    for (int g = 0; g < G; g++) for (size_t k = 0; k < plan[g].size(); k++) out->n_pairs += jobs[g].h_pairs[k] / 2;
    for (int64_t c = 0; c < C; c++) out->n_chains_ok += out->status[c] == AHS_CHAIN_OK;
    // ---- timings (max over devices) and byte counts
    int bits = 2;
    for (int g = 0; g < G; g++) {
        float ms7[7]; int launches = 0;
        CK(cudaSetDevice(devs[g]));
        jobs[g].times(ms7, launches);
        out->ms_h2d = std::max(out->ms_h2d, jobs[g].h2d); out->ms_d2h = std::max(out->ms_d2h, jobs[g].d2h);
        out->ms_project = std::max(out->ms_project, ms7[0]); out->ms_rows = std::max(out->ms_rows, ms7[1]); out->ms_score = std::max(out->ms_score, ms7[2]);
        out->ms_cluster = std::max(out->ms_cluster, ms7[3]); out->ms_consensus = std::max(out->ms_consensus, ms7[4]); out->ms_thread = std::max(out->ms_thread, ms7[5]);
        out->ms_total_device = std::max(out->ms_total_device, ms7[6]);
        out->n_launches += launches;
        for (auto& pl : jobs[g].pls) if (pl.sz.C) bits = std::max(bits, (int)pl.d.bits);
    }
    {   // algorithmic bytes, SURVEY.md §8d: each datum crosses HBM once
        const double code_bytes = bits / 8.0;
        const int64_t cells = out->n_cells;
        out->bytes_project = 4 * sz.NEN + 4 * sz.NAN_ + 8 * sz.NE + (int64_t)(code_bytes * cells) + 12 * NFt;
        out->bytes_score = (int64_t)(code_bytes * cells) + 12 * NFt + 4 * out->n_pairs;
        out->bytes_consensus = (int64_t)(code_bytes * cells) + 16 * NFt + 5 * NPt * p;   // k_pos ~ ploidy retained clusters
    }
}

}  // namespace ahs

using namespace ahs;

extern "C" {

int ahs_abi_version(void) { return AHS_ABI_VERSION; }

void ahs_get_limits(ahs_limits* out) {
    if (!out) return;
    memset(out, 0, sizeof(*out));
    out->max_ploidy = MAX_PLOIDY; out->max_alleles = MAX_ALLELES; out->max_reads_cluster = MAX_READS_CLUSTER; out->max_positions = MAX_POSITIONS;
    out->max_clusters_position = K3_CAP;
}

int ahs_device_count(void) { int n = 0; if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; } return n; }

const char* ahs_last_error(void) { return g_err; }

double ahs_chain_cost(int64_t n_bubbles, int64_t n_entries, int64_t n_entry_nodes, int ploidy) {
    // SM-milliseconds of one chain, calibrated on B200 from the per-class launch times of cfg2 and the stage times of the other
    // configurations (DESIGN.md section 8).  nf = final reads ~ 0.7 x entries.  Projection / rows / scoring / consensus stream
    // the alignment nodes; cluster editing dominates: ~nf^2 in the shared-memory kernel (its parallel width grows with the
    // pairs), ~nf^3 up to 1,024 reads, ~nf x neighbourhood above; the threading DP is per position x states.  The nf^3 regime
    // predates k_cluster_sparse, which now takes every chain above CC_MAXN reads: it was calibrated on that kernel's dense
    // predecessor and is kept as it is, because it sets the range count (ranges_of_share) and the device cuts (plan_devices).
    const double nf = 0.7 * (double)n_entries;
    double cluster;
    if (nf <= 160.0) cluster = 2.9e-5 * nf * nf;
    else if (nf <= 1024.0) cluster = 9e-7 * nf * nf * nf;
    else cluster = 9e-7 * 1024.0 * 1024.0 * 1024.0 + 0.3 * (nf - 1024.0);
    double S = 1; for (int i = 0; i < ploidy && i < 4; i++) S *= 2 * ploidy;
    if (ploidy > 4) S = 1716;
    return 1e-5 * (double)n_entry_nodes + cluster + 1e-7 * (double)n_bubbles * S;
}

int ahs_plan_shares(const double* chain_cost, int64_t n_chains, int n_parts, int64_t* cuts) {
    return guarded("ahs_plan_shares", [&]() {
        if (!cuts || n_parts < 1 || n_chains < 0 || (n_chains > 0 && !chain_cost)) throw ArgFail{"ahs_plan_shares: bad arguments"};
        std::vector<double> pre((size_t)n_chains + 1, 0.0);
        for (int64_t c = 0; c < n_chains; c++) {
            if (!(chain_cost[c] >= 0.0)) throw ArgFail{"ahs_plan_shares: negative or NaN cost"};
            pre[c + 1] = pre[c] + chain_cost[c];
        }
        const std::vector<int64_t> r = balanced_contiguous_cuts(pre, n_parts);
        for (int g = 0; g <= n_parts; g++) cuts[g] = r[g];
    });
}

int ahs_phase_batch(const ahs_batch_in* in, ahs_batch_out* out, int device) {
    return guarded("ahs_phase_batch", [&]() { phase_on_devices(in, nullptr, out, &device, 1, 0, 0); });
}

int ahs_phase_batch_resident(const ahs_batch_in* in, ahs_batch_out* out, int device, int warmup, int iters) {
    return guarded("ahs_phase_batch_resident", [&]() { phase_on_devices(in, nullptr, out, &device, 1, warmup < 0 ? 0 : warmup, iters < 1 ? 1 : iters); });
}

int ahs_phase_batch_multi(const ahs_batch_in* in, ahs_batch_out* out, const int* device_ids, int n_devices) {
    return guarded("ahs_phase_batch_multi", [&]() { phase_on_devices(in, nullptr, out, device_ids, n_devices, 0, 0); });
}

int ahs_phase_batch_genotyped(const ahs_batch_in* in, const uint8_t* allele_dosage, ahs_batch_out* out, const int* device_ids, int n_devices) {
    return guarded("ahs_phase_batch_genotyped", [&]() { phase_on_devices(in, allele_dosage, out, device_ids, n_devices, 0, 0); });
}

int ahs_debug_std_sort(int32_t* keys, int32_t* values, int32_t n, int descending, int device) {
    return guarded("ahs_debug_std_sort", [&]() {
        if (n < 0 || (n > 0 && (!keys || !values))) throw ArgFail{"null array"};
        Ctx* cx = get_ctx(device);
        std::lock_guard<std::mutex> g(cx->mu);
        CK(cudaSetDevice(device));
        if (n == 0) return;
        int32_t *dk = nullptr, *dv = nullptr;
        CK(cudaMalloc(&dk, (size_t)n * 4)); CK(cudaMalloc(&dv, (size_t)n * 4));
        CK(cudaMemcpy(dk, keys, (size_t)n * 4, cudaMemcpyHostToDevice)); CK(cudaMemcpy(dv, values, (size_t)n * 4, cudaMemcpyHostToDevice));
        k_debug_std_sort<<<1, 1>>>(dk, dv, n, descending);
        cudaError_t e = cudaDeviceSynchronize();
        if (e == cudaSuccess) { CK(cudaMemcpy(keys, dk, (size_t)n * 4, cudaMemcpyDeviceToHost)); CK(cudaMemcpy(values, dv, (size_t)n * 4, cudaMemcpyDeviceToHost)); }
        cudaFree(dk); cudaFree(dv);
        CK(e);
    });
}

int ahs_warmup(int device, uint64_t device_bytes, uint64_t pinned_bytes) {
    return guarded("ahs_warmup", [&]() {
        Ctx* cx = get_ctx(device);
        std::lock_guard<std::mutex> g(cx->mu);
        CK(cudaSetDevice(device));
        if (cx->out_busy) return;                          // a result is outstanding: its pools must not move
        auto reserve = [](Pool& p, uint64_t bytes) {
            size_t have = 0; for (auto& c : p.chunks) have = std::max(have, c.cap);
            if (bytes > have) { p.alloc((size_t)bytes); p.reset(); }
        };
        reserve(cx->dev, device_bytes);
        reserve(cx->outp, pinned_bytes);                   // results (zero-copy output arrays)
        reserve(cx->pin, pinned_bytes ? (size_t)64 << 20 : 0);   // staging of the per-chain offset arrays
    });
}

int ahs_pin_host(const void* ptr, uint64_t bytes) {
    if (!ptr || !bytes) return AHS_OK;
    cudaError_t e = cudaHostRegister(const_cast<void*>(ptr), bytes, cudaHostRegisterPortable);
    if (e != cudaSuccess && e != cudaErrorHostMemoryAlreadyRegistered) { set_err("ahs_pin_host: %s", cudaGetErrorString(e)); cudaGetLastError(); return AHS_ERR_CUDA; }
    cudaGetLastError();
    return AHS_OK;
}
int ahs_unpin_host(const void* ptr) {
    if (!ptr) return AHS_OK;
    cudaError_t e = cudaHostUnregister(const_cast<void*>(ptr));
    cudaGetLastError();
    return e == cudaSuccess ? AHS_OK : AHS_ERR_CUDA;
}

void ahs_free_out(ahs_batch_out* out) {
    if (!out) return;
    if (out->read_off) {
        // the arrays live in the page-locked result pool of one device context: find it by address
        Ctx* owner = nullptr;
        {
            std::lock_guard<std::mutex> g(g_ctx_mu);
            for (auto* c : g_ctx) if (c && !owner)
                for (auto& ch : c->outp.chunks) if ((char*)out->read_off >= ch.p && (char*)out->read_off < ch.p + ch.cap) owner = c;
        }
        if (owner) { std::lock_guard<std::mutex> g(owner->mu); owner->out_busy = false; }
    }
    memset(out, 0, sizeof(*out));
}

}  // extern "C"
