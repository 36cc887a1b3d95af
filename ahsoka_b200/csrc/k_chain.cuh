// k_chain.cuh — read-pair scoring and cluster editing out of shared memory, one thread block per chain.
//
// Replaces ReadScoring::scoreReadsetLocal + ClusterEditingSolver::run (call sites reference
// src/alignmentstoreadset.cpp:308-315; algorithms: oracle/core/phase_core.hpp rules R1 and R2) for
// chains with at most CC_MAXN final reads — every chain of BASELINE config 2.  Larger chains take
// the HBM-resident path (k_read_rates / k_pair_scores / k_cluster_sparse).
//
//   k_score_chain    K2: reads the packed allele rows (code_bytes per cell) + 8 B of row descriptors per
//                    read, writes one int32 Q10 weight per read pair (upper triangle, row-major): exactly
//                    the algorithmic traffic of SURVEY §8d.
//   k_cluster_chain  reads those 4 B per pair once, writes 4 B of cluster label per read.
// (Two kernels rather than one: the greedy loop of cluster editing is instruction-issue bound and its
// code must stay inside the 32 KB L1.5 instruction cache; the pair weights cost 0.07 ms of HBM time.)
//
// k_cluster_chain:
// Where the state lives
//   registers  every thread OWNS up to PER (8 or 12) read pairs ("slots"): key = (a << 8 | b), a < b, plus
//              the pair's induced costs icf / icp (rule R2).  Scans for the best candidate and all
//              induced-cost updates are register arithmetic by the owner; a slot only ever dies
//              (merge / forbid) or is relabelled in place ((b,x) becomes (a,x) when b merges into a),
//              so no list is ever appended to.
//   shared     W[n][ns] int32, the symmetric weight matrix (0 = no edge, CC_FORB = forbidden), row
//              stride ns odd -> conflict-free row AND column walks; per-node records of the current
//              merge (old weights to a and b, merged weight), the fresh induced costs of the merged
//              node's pairs, and per-node bit masks of the edges flagged in a forbid round.
// int32 is exact: every weight and induced cost is bounded by the sum of |w| over the chain's pairs
// <= 16290 * 2^17 < 2^31 for n <= 181.
//
// The greedy loop is sequential by definition (argmax -> merge or forbid).  One step = a few
// barrier-separated passes in which every thread walks its own slots; the argmax of the next step
// is folded into the last pass of the current one.  Runs of single-edge forbids are batched EXACTLY
// (see "round" below).
#pragma once
#include "common.cuh"
#include "device_batch.cuh"
#include "k_score.cuh"
#include "k_select.cuh"

namespace ahs {

constexpr int CC_MAXN = 160;
constexpr int32_t CC_FORB = -0x7fffffff;          // forbidden edge inside this kernel (-CC_FORB is representable)
constexpr uint32_t CC_POS = 1u << 31;             // slot flag: weight > 0 (sign bit: see CCBest::consider)
constexpr uint32_t CC_FLAG = 1u << 17;            // slot flag: edge was forbidden in a round (tentatively, then for good)
constexpr uint32_t CC_DEAD = 1u << 18;            // slot flag: no candidate pair in this slot
constexpr uint32_t CC_GONE = CC_FLAG | CC_DEAD;

__host__ __device__ inline int cc_ns(int nmax) { return nmax | 1; }
__host__ __device__ inline int cc_mw(int nmax) { return (nmax + 31) / 32; }

__host__ __device__ inline size_t cc_smem_bytes(int nmax, int nthreads) {
    size_t b = (size_t)nmax * cc_ns(nmax) * 4 * 2;        // W, D
    b += (size_t)nmax * 16;                               // node records {wa, wb, nw, -}
    b += (size_t)nmax * 4 * 2;                            // frF, frP
    b += (size_t)nmax * cc_mw(nmax) * 4;                  // fmask
    b += (size_t)(nthreads / 32) * 8 * 4 * 2;             // reduction scratch, double buffered
    b += 64;                                              // scalars
    b += (size_t)nmax * 5;                                // alist, apos, label, active, nodefl (u8 each)
    return (b + 15) & ~(size_t)15;
}

__device__ __forceinline__ unsigned long long cc_globaltimer() {
    unsigned long long t; asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t)); return t;
}
// tf(x,y) = min(x,y) if both positive else 0;  tp(x,y) = min(pos, |neg|) if the signs differ else 0  (rule R2)
__device__ __forceinline__ int cc_tf(int x, int y) { return max(min(x, y), 0); }
__device__ __forceinline__ int cc_tp(int x, int y) { const int lo = min(x, y), hi = max(x, y); return max(min(hi, -lo), 0); }

struct CCBest {          // running maxima of one thread / of the block: max icf, max icp, max icp over positive edges
    int M, maxP, maxPpos, live;                         // live: slots seen by this thread (not reduced)
    __device__ __forceinline__ void clear() { M = -1; maxP = -1; maxPpos = -1; live = 0; }
    __device__ __forceinline__ void consider(uint32_t key, int f, int p) {
        M = max(M, f); maxP = max(maxP, p);
        const int pos = (int)key >> 31;                 // all ones for a positive edge
        maxPpos = max(maxPpos, (p & pos) | ~pos);       // p, or -1 for a negative edge
        live++;
    }
};

// block-wide maxima.  Contains one barrier.
template <int NT>
__device__ __forceinline__ CCBest cc_reduce(const CCBest& b, int32_t* red, int tid, int& phase) {
    constexpr int NW = NT / 32;
    CCBest w;
    w.M = __reduce_max_sync(0xffffffffu, b.M); w.maxP = __reduce_max_sync(0xffffffffu, b.maxP); w.maxPpos = __reduce_max_sync(0xffffffffu, b.maxPpos);
    if (NW == 1) { __syncthreads(); return w; }
    int32_t* r = red + phase * (NW * 4);
    if ((tid & 31) == 0) { int32_t* q = r + (tid >> 5) * 4; q[0] = w.M; q[1] = w.maxP; q[2] = w.maxPpos; }
    __syncthreads();
    const int lane = tid & 31;
    CCBest o; o.clear();
    if (lane < NW) { const int32_t* q = r + lane * 4; o.M = q[0]; o.maxP = q[1]; o.maxPpos = q[2]; }
    phase ^= 1;
    w.M = __reduce_max_sync(0xffffffffu, o.M); w.maxP = __reduce_max_sync(0xffffffffu, o.maxP); w.maxPpos = __reduce_max_sync(0xffffffffu, o.maxPpos);
    return w;
}

// smallest pair key (a << 8 | b) among the slots whose value equals the block maximum: the tie rule of rule R2.
// `mine` = smallest matching key of this thread (0xffff if none).  Contains one barrier.
__device__ __forceinline__ int cc_min_key(int mine, int32_t* cell, int tid, int& kphase) {
    const int wmin = __reduce_min_sync(0xffffffffu, mine);
    if ((tid & 31) == 0 && wmin < 0xffff) atomicMin(&cell[kphase], wmin);
    if (tid == 0) cell[kphase ^ 1] = 0xffff;            // last read at least one barrier ago
    __syncthreads();
    const int r = cell[kphase];
    kphase ^= 1;
    return r;
}

// ascending bitonic sort of 32*KPL keys (uint32_t or uint64_t) held KPL per lane (element e = s*32 + lane)
template <int KPL, class T>
__device__ __forceinline__ void warp_sort(T (&v)[KPL], int lane) {
#pragma unroll
    for (int kk = 2; kk <= 32 * KPL; kk <<= 1) {
#pragma unroll
        for (int jj = kk >> 1; jj > 0; jj >>= 1) {
            if (jj >= 32) {
#pragma unroll
                for (int s = 0; s < KPL; s++) {
                    if ((s & (jj >> 5)) == 0) {
                        const int s2 = s | (jj >> 5);
                        const bool up = ((s * 32) & kk) == 0;          // lane bits are below jj >= 32 <= kk/2
                        const T a = v[s], b = v[s2];
                        if ((a > b) == up) { v[s] = b; v[s2] = a; }
                    }
                }
            } else {
#pragma unroll
                for (int s = 0; s < KPL; s++) {
                    const bool up = ((s * 32 + lane) & kk) == 0;
                    const T other = __shfl_xor_sync(0xffffffffu, v[s], jj);
                    const bool keep_min = ((lane & jj) == 0) == up;
                    v[s] = keep_min ? (other < v[s] ? other : v[s]) : (other > v[s] ? other : v[s]);
                }
            }
        }
    }
}

// Rule R1's pooling for one read: the m partner keys in ws[0..m) (any order) are sorted as 32*K2 >= m keys, the `cut`
// lowest rates are pooled as same-haplotype pairs, the rest as different-haplotype pairs.  K_BITS / N_SHIFT / MASK give
// the (k, n) fields of a key.
template <int K2, class T, int N_SHIFT, int MASK>
__device__ __forceinline__ void cs_pool(const T* __restrict__ ws, int m, int cut, int lane, int& Ks, int& Ns, int& Kd, int& Nd) {
    T v[K2];
#pragma unroll
    for (int s = 0; s < K2; s++) v[s] = s * 32 + lane < m ? ws[s * 32 + lane] : (T)~(T)0;
    warp_sort<K2>(v, lane);
#pragma unroll
    for (int s = 0; s < K2; s++) if (s * 32 + lane < m) {
        const int kq = (int)(v[s] & (T)MASK), nq = (int)((v[s] >> N_SHIFT) & (T)MASK);
        if (s * 32 + lane < cut) { Ks += kq; Ns += nq; } else { Kd += kq; Nd += nq; }
    }
}
template <int KPL, class T, int N_SHIFT, int MASK>
__device__ __forceinline__ void cs_pool_any(const T* __restrict__ ws, int m, int cut, int lane, int& Ks, int& Ns, int& Kd, int& Nd) {
    if (m <= 32) cs_pool<1, T, N_SHIFT, MASK>(ws, m, cut, lane, Ks, Ns, Kd, Nd);
    else if (KPL >= 2 && m <= 64) cs_pool<(KPL >= 2 ? 2 : 1), T, N_SHIFT, MASK>(ws, m, cut, lane, Ks, Ns, Kd, Nd);
    else if (KPL >= 8 && m <= 128) cs_pool<(KPL >= 8 ? 4 : 1), T, N_SHIFT, MASK>(ws, m, cut, lane, Ks, Ns, Kd, Nd);
    else cs_pool<KPL, T, N_SHIFT, MASK>(ws, m, cut, lane, Ks, Ns, Kd, Nd);
}

// ------------------------------------------------------------------------------------------------
// K2: read-pair scoring of one chain per block (rule R1).  Wout[cw_off[c] + pair number] = Q10 weight,
// pair number = position of (x,y), x < y, in the row-major upper triangle.
//
// Reads are sorted by first position, so the partners y > x of read x form the index band first[y] <= last[x]:
// only the band is scored (16 lanes per row x, lanes over y; no pair-number arithmetic).
//   pass 1  every band pair: overlap n and disagreements k by AND / XOR / popcount over the words of the shared
//           span.  n <= 254 ("narrow": the chain's longest read spans < 255 bubbles): the pair's ORDER KEY
//           floor(65534 k/n) << 16 | n << 8 | k goes into both triangles of KEY[n][n|1] and (n << 8 | k) into NK16[pair].
//           Distinct rates with denominators <= 255 differ by more than 1/65534, so the 32-bit key orders exactly like
//           rule R1's (k/n, n, k); the division is a multiplication by a reciprocal table.
//   pass 2  local rates, one warp per read: the valid keys of the read's row are compacted (ballot) and sorted in
//           registers (bitonic, 32 / 64 / 128 / 32 KPL keys as needed); the cut = max(1, m/p) lowest are pooled as
//           same-haplotype pairs, the rest as different-haplotype pairs.  (A one-thread-per-read radix selection —
//           k_select.cuh, kept with its host harness — needs 36 % fewer instructions but leaves most warps of the
//           block waiting at the barrier: measured 2.1 ms against 1.9 ms for this pass structure on cfg2.)
//   pass 3  fixed-point log-likelihood ratio of every band pair from NK16 and the reads' rates; zeros elsewhere.
// Chains with a read of 255+ bubbles ("wide") keep (n << 16 | k) in KEY and rank by exact cross products.
// ------------------------------------------------------------------------------------------------
constexpr int CS_GROUP = 16;                          // lanes per row in the pair passes

__host__ __device__ inline size_t cs_smem_bytes(int nmax, int nt) {
    size_t b = (size_t)nmax * cc_ns(nmax) * 4;                          // KEY
    b += ((size_t)nmax * (nmax - 1) / 2 * 2 + 15) & ~(size_t)15;       // NK16
    b += (size_t)(nt / 32) * nmax * 4;                                  // per-warp scratch of the rate sort: the compacted keys of one read
    b += (size_t)nmax * 4 * 2 + (size_t)nmax * 2 * 2 + 16;              // first, last, es, ed
    b += 256 * 4 + 64;                                                  // reciprocals, scalars
    return (b + 15) & ~(size_t)15;
}

template <int BITS>
__device__ __forceinline__ void span_nk(const uint32_t* __restrict__ rx, const uint32_t* __restrict__ ry, int lo_b, int hi_b, int& n, int& k) {
    constexpr int PW = 32 / BITS;
    n = 0; k = 0;
    const int w1 = hi_b / PW;
    for (int w = lo_b / PW; w <= w1; w += 2) {                         // two words per trip: four independent loads in flight
        const bool two = w + 1 <= w1;
        const uint32_t x0 = __ldg(rx + w), y0 = __ldg(ry + w);
        const uint32_t x1 = two ? __ldg(rx + w + 1) : 0u, y1 = two ? __ldg(ry + w + 1) : 0u;
        word_nk<BITS>(x0, y0, n, k); word_nk<BITS>(x1, y1, n, k);
    }
}

template <int BITS, int NT, int KPL>
__global__ void __launch_bounds__(NT) k_score_chain(DB d, const int32_t* __restrict__ chains, int n_list, int nmax,
                                                    int32_t* __restrict__ work_counter) {
    extern __shared__ __align__(16) unsigned char cc_sm[];
    constexpr int NW = NT / 32;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int ns = cc_ns(nmax);
    uint32_t* KEY; uint16_t* NK16; uint32_t* hist; int32_t *first, *last, *scal; uint32_t* rcp; uint16_t *es, *ed;
    {
        unsigned char* p = cc_sm;
        KEY = (uint32_t*)p; p += (size_t)nmax * ns * 4;
        NK16 = (uint16_t*)p; p += ((size_t)nmax * (nmax - 1) / 2 * 2 + 15) & ~(size_t)15;
        hist = (uint32_t*)p + (size_t)wid * nmax; p += (size_t)NW * nmax * 4;      // this warp's sort scratch
        first = (int32_t*)p; p += nmax * 4; last = (int32_t*)p; p += nmax * 4;
        es = (uint16_t*)p; p += nmax * 2; ed = (uint16_t*)p; p += nmax * 2; p = (unsigned char*)(((uintptr_t)p + 15) & ~(uintptr_t)15);
        rcp = (uint32_t*)p; p += 256 * 4;
        scal = (int32_t*)p;
    }
    // reciprocal table, once per block (k_select.cuh)
    for (int x = tid; x < 256; x += NT) rcp[x] = cs_rcp((uint32_t)x);
    const unsigned gm = grp_mask<CS_GROUP>();
    const int gl = lane % CS_GROUP, grp = tid / CS_GROUP;
    constexpr int NG = NT / CS_GROUP;
    int64_t pairs_total = 0;
    (void)work_counter; (void)scal;
    // static round robin over the class's chains (they are sorted by read count: neighbours cost the same); no work counter,
    // so a block's next chain is known ahead and its descriptors are already on their way when the current chain ends
    for (int item = blockIdx.x; item < n_list; item += gridDim.x) {
        const int c = chains[item];
        const int64_t f0 = d.frow_off[c];
        const int n = (int)(d.frow_off[c + 1] - f0);
        __syncthreads();                                              // the previous chain's last pass is done with the shared arrays
        const int words = d.ch_words[c];
        const uint32_t* rows = d.codes + d.code_off[c];
        int32_t* Wout = d.W + d.cw_off[c];
        const bool narrow = d.ch_maxspan[c] < 254;                    // overlaps n <= span <= 254
        for (int x = tid; x < n; x += NT) { first[x] = d.fr_first[f0 + x]; last[x] = d.fr_last[f0 + x]; }
        for (int x = tid; x < n * ns; x += NT) KEY[x] = CS_INVALID;
        __syncthreads();
        // ---- pass 1: counts of the band pairs
        for (int x = grp; x < n - 1; x += NG) {
            const int lx = last[x];
            const uint32_t* rx = rows + (int64_t)x * words;
            const int rowbase = ((x * (2 * n - x - 1)) >> 1) - (x + 1);          // pair number of (x,y) = rowbase + y
            for (int y0 = x + 1; y0 < n; y0 += CS_GROUP) {
                const int y = y0 + gl;
                const bool valid = y < n;
                const int fy = valid ? first[y] : INT32_MAX;
                const bool inband = fy <= lx;
                if (inband) {
                    int nn, kk; span_nk<BITS>(rx, rows + (int64_t)y * words, fy, min(lx, last[y]), nn, kk);
                    if (narrow) {
                        NK16[rowbase + y] = (uint16_t)((nn << 8) | kk);
                        if (nn > 0) { const uint32_t key = cs_order_key((uint32_t)nn, (uint32_t)kk, rcp[nn]); KEY[x * ns + y] = key; KEY[y * ns + x] = key; }
                    } else if (nn > 0) { const uint32_t nk = ((uint32_t)nn << 16) | (uint32_t)kk; KEY[x * ns + y] = nk; KEY[y * ns + x] = nk; }
                    else KEY[x * ns + y] = 0u;                                    // wide: in band, no shared position (pass 3 reads KEY)
                }
                if (!__any_sync(gm, inband)) break;                               // first[] ascends: the rest of the row is out of band too
            }
        }
        __syncthreads();
        // ---- pass 2: local rates
        if (narrow) {
            const unsigned lt = (1u << lane) - 1u;
            for (int i = wid; i < n; i += NW) {
                const uint32_t* row = KEY + i * ns;
                int m = 0, Ks = 0, Ns = 0, Kd = 0, Nd = 0;
#pragma unroll
                for (int s5 = 0; s5 < KPL; s5++) {
                    const int j = s5 * 32 + lane;
                    const uint32_t key = j < n ? row[j] : CS_INVALID;
                    const uint32_t bal = __ballot_sync(0xffffffffu, key != CS_INVALID);
                    if (key != CS_INVALID) hist[m + __popc(bal & lt)] = key;
                    m += __popc(bal);
                }
                __syncwarp();
                if (m > 0) cs_pool_any<KPL, uint32_t, 8, 0xff>(hist, m, max(1, m / d.ploidy), lane, Ks, Ns, Kd, Nd);
                __syncwarp();                                   // the scratch is rewritten for the warp's next read
                uint32_t es_i = 0, ed_i = 0;
                if (m > 0) {
                    Ks = warp_sum_i32(Ks); Ns = warp_sum_i32(Ns); Kd = warp_sum_i32(Kd); Nd = warp_sum_i32(Nd);
                    es_i = ((uint32_t)Ks * 1024u + (uint32_t)Ns / 2u) / (uint32_t)Ns;          // sums of < CC_MAXN values <= 255: 32 bits
                    ed_i = Nd > 0 ? ((uint32_t)Kd * 1024u + (uint32_t)Nd / 2u) / (uint32_t)Nd : es_i;
                }
                if (lane == 0) { es[i] = (uint16_t)es_i; ed[i] = (uint16_t)ed_i; pairs_total += m; }
            }
        } else if (tid < n) {
            // wide (a read of 255+ bubbles): exact order (k_a n_b < k_b n_a, then n, then k) by counting, one thread per read, O(m^2)
            const uint32_t* row = KEY + tid * ns;
            int Ks = 0, Ns = 0, Kd = 0, Nd = 0, m = 0;
            for (int j = 0; j < n; j++) { const uint32_t v = row[j]; m += (v != CS_INVALID && v != 0u) ? 1 : 0; }
            const int cut = m ? max(1, m / d.ploidy) : 0;
            for (int a = 0; a < n && m; a++) {
                const uint32_t va = row[a];
                if (va == CS_INVALID || va == 0u) continue;
                const long long na = va >> 16, ka = va & 0xffffu;
                int r = 0;
                for (int b = 0; b < n; b++) {
                    const uint32_t vb = row[b];
                    if (vb == CS_INVALID || vb == 0u) continue;
                    const long long nb = vb >> 16, kb = vb & 0xffffu;
                    const long long l = kb * na, rr = ka * nb;                // b before a ?
                    const bool less = l != rr ? l < rr : (nb != na ? nb < na : (kb != ka ? kb < ka : b < a));
                    r += less ? 1 : 0;
                }
                if (r < cut) { Ks += (int)ka; Ns += (int)na; } else { Kd += (int)ka; Nd += (int)na; }
            }
            uint32_t es_i = 0, ed_i = 0;
            if (m > 0) {
                es_i = (uint32_t)(((int64_t)Ks * 1024 + Ns / 2) / Ns);
                ed_i = Nd > 0 ? (uint32_t)(((int64_t)Kd * 1024 + Nd / 2) / Nd) : es_i;
            }
            es[tid] = (uint16_t)es_i; ed[tid] = (uint16_t)ed_i;
            pairs_total += m;
        }
        __syncthreads();
        // ---- pass 3: pair weights (fixed-point log likelihood ratio), 4 B per pair to HBM
        for (int x = grp; x < n - 1; x += NG) {
            const int lx = last[x];
            const int esx = es[x], edx = ed[x];
            const int rowbase = ((x * (2 * n - x - 1)) >> 1) - (x + 1);
            for (int y = x + 1 + gl; y < n; y += CS_GROUP) {
                int w = 0;
                if (first[y] <= lx) {
                    int nn, kk;
                    if (narrow) { const int nk = NK16[rowbase + y]; nn = nk >> 8; kk = nk & 255; }
                    else { const uint32_t nk = KEY[x * ns + y]; nn = (int)(nk >> 16); kk = (int)(nk & 0xffffu); }      // this triangle is not permuted in the wide path
                    if (nn > 0) {
                        int e1 = (esx + es[y]) >> 1, e2 = (edx + ed[y]) >> 1;
                        e1 = min(max(e1, 10), 460);
                        e2 = min(max(e2, e1 + 51), 972);
                        const int64_t s20 = (int64_t)kk * (int)(__ldg(d.ln + e1) - __ldg(d.ln + e2)) + (int64_t)(nn - kk) * (int)(__ldg(d.ln1 + e1) - __ldg(d.ln1 + e2));      // |ln| 2^20 < 2^23: the differences fit 32 bits
                        w = narrow ? (int)(s20 >> 10) : (int)max(min(s20 >> 10, (int64_t)W_CLAMP), (int64_t)-W_CLAMP);      // narrow: |s20| < 2^34, the quotient fits 32 bits
                        w = min(max(w, -W_CLAMP), W_CLAMP);
                    }
                }
                Wout[rowbase + y] = w;
            }
        }
    }
    pairs_total = warp_sum_i64(pairs_total);
    if (lane == 0 && pairs_total) atomicAdd((unsigned long long*)d.tot_pairs, (unsigned long long)pairs_total);
}

// resident blocks per SM the register allocation is held to (~64 registers per thread: 24 of them are the slots)
__host__ __device__ constexpr int cc_min_blocks(int nt, int per) {
    // registers per thread ~ 40 + 3 per slot
    return per > 8 ? (nt <= 96 ? 8 : nt <= 128 ? 6 : nt <= 192 ? 4 : nt <= 256 ? 3 : nt <= 384 ? 2 : 1)
         : per <= 4 ? (nt <= 32 ? 32 : nt <= 64 ? 20 : nt <= 128 ? 10 : nt <= 192 ? 6 : nt <= 256 ? 5 : nt <= 384 ? 3 : nt <= 512 ? 2 : 1)
                    : (nt <= 32 ? 32 : nt <= 64 ? 18 : nt <= 96 ? 12 : nt <= 128 ? 9 : nt <= 192 ? 6 : nt <= 256 ? 4 : nt <= 384 ? 3 : nt <= 512 ? 2 : 1);
}

// lanes that share one node x in the fresh-cost pass of a merge (threads / G >= largest n of the block size's classes)
__host__ __device__ constexpr int cc_fresh_g(int nt, int per = 8) { return per > 8 ? (nt <= 64 ? 1 : nt < 512 ? 2 : 4) : nt <= 32 ? 1 : nt <= 192 ? 2 : nt <= 768 ? 4 : 8; }
static_assert(CC_MAXN <= 160, "k_cluster_chain walks rows in five 32-lane strides");

// ------------------------------------------------------------------------------------------------
// cluster editing of one chain per block (rule R2)
// ------------------------------------------------------------------------------------------------
template <int NT, int PER>
__global__ void __launch_bounds__(NT, cc_min_blocks(NT, PER)) k_cluster_chain(DB d, const int32_t* __restrict__ chains, int n_list, int nmax,
                                                                         int32_t* __restrict__ work_counter, int32_t* __restrict__ scratch) {
    extern __shared__ __align__(16) unsigned char cc_sm[];
    constexpr int NW = NT / 32;
    const int tid = threadIdx.x, lane = tid & 31, wid = tid >> 5;
    const int ns = cc_ns(nmax), mw = cc_mw(nmax);
    int32_t *W, *D; int4* node; int32_t *frF, *frP; uint32_t* fmask; int32_t *red, *scal;
    uint8_t *alist, *apos, *label, *active, *nodefl;
    {
        unsigned char* p = cc_sm;
        node = (int4*)p; p += (size_t)nmax * 16;
        W = (int32_t*)p; p += (size_t)nmax * ns * 4;
        D = (int32_t*)p; p += (size_t)nmax * ns * 4;
        frF = (int32_t*)p; p += nmax * 4; frP = (int32_t*)p; p += nmax * 4;
        fmask = (uint32_t*)p; p += (size_t)nmax * mw * 4;
        red = (int32_t*)p; p += NW * 8 * 4 * 2;
        scal = (int32_t*)p; p += 64;                  // [0] active nodes, [1] edges flagged in the round, [3] work item
        alist = p; p += nmax; apos = p; p += nmax; label = p; p += nmax; active = p; p += nmax; nodefl = p; p += nmax;
    }
    constexpr bool WIDE5 = NT == 1024 && PER > 8;      // the classes above 128 reads: rows are walked in five 32-lane strides
    int phase = 0, kphase = 0;
    uint32_t key[PER]; int F[PER], P[PER];
    int32_t* scr = scratch + ((size_t)blockIdx.x * NW + wid) * (32 * PER * 3);       // this warp's packing area (global, L2)
    const unsigned lt = (1u << lane) - 1u;
    while (true) {
        __syncthreads();
        if (tid == 0) scal[3] = atomicAdd(work_counter, 1);
        __syncthreads();
        const int item = scal[3];
        if (item >= n_list) break;
        const int c = chains[item];
        const int64_t f0 = d.frow_off[c];
        const int n = (int)(d.frow_off[c + 1] - f0);
        const int tri = n * (n - 1) / 2;
        const int32_t* Win = d.W + d.cw_off[c];
        for (int x = tid; x < n; x += NT) {
            active[x] = 1; label[x] = (uint8_t)x; alist[x] = (uint8_t)x; apos[x] = (uint8_t)x; nodefl[x] = 0;
            W[x * ns + x] = 0;
            for (int m = 0; m < mw; m++) fmask[x * mw + m] = 0;
        }
        if (tid == 0) { scal[0] = n; scal[1] = 0; scal[4] = 0xffff; scal[5] = 0xffff; kphase = 0; }
        else kphase = 0;
        int x0 = 0, y0 = 1;
        if (tid < tri) {
            const float tn = (float)(2 * n - 1);
            int x = (int)((tn - sqrtf(tn * tn - 8.0f * (float)tid)) * 0.5f);
            x = max(0, min(x, n - 2));
            while (x > 0 && ((x * (2 * n - x - 1)) >> 1) > tid) x--;
            while ((((x + 1) * (2 * n - x - 2)) >> 1) <= tid) x++;
            x0 = x; y0 = x + 1 + tid - ((x * (2 * n - x - 1)) >> 1);
        }
        // weights: 4 B per pair from HBM into the symmetric matrix
        {
            int x = x0, y = y0;
            for (int ti = tid; ti < tri; ti += NT) {
                const int w = __ldg(Win + ti);
                W[x * ns + y] = w; W[y * ns + x] = w;
                if (ti + NT < tri) { y += NT; while (y >= n) { y = y - n + x + 2; x++; } }
            }
        }
        __syncthreads();
        // initial induced costs of the thread's own pairs (W[x][x] = 0 makes the third nodes t = x, y contribute
        // nothing), parked in D so that this loop need not be unrolled over the register slots
        {
            int x = x0, y = y0;
            for (int ti = tid; ti < tri; ti += NT) {
                const int32_t* rx = W + x * ns; const int32_t* ry = W + y * ns;
                const int w = rx[y];
                if (w != 0) {
                    int f = max(w, 0), p = max(-w, 0);
                    for (int t = 0; t < n; t++) { const int wx = rx[t], wy = ry[t]; f += cc_tf(wx, wy); p += cc_tp(wx, wy); }
                    D[ti] = f; D[tri + ti] = p;
                }
                if (ti + NT < tri) { y += NT; while (y >= n) { y = y - n + x + 2; x++; } }
            }
        }
        CCBest mine; mine.clear();
        {
            int x = x0, y = y0;
#pragma unroll
            for (int k = 0; k < PER; k++) {
                key[k] = CC_DEAD; F[k] = 0; P[k] = 0;
                const int ti = k * NT + tid;
                if (ti < tri) {
                    const int w = W[x * ns + y];
                    if (w != 0) {
                        key[k] = (uint32_t)((x << 8) | y) | (w > 0 ? CC_POS : 0u); F[k] = D[ti]; P[k] = D[tri + ti];
                        mine.consider(key[k], F[k], P[k]);
                    }
                    if (ti + NT < tri) { y += NT; while (y >= n) { y = y - n + x + 2; x++; } }
                }
            }
        }
        CCBest so = cc_reduce<NT>(mine, red, tid, phase);
        bool force_single = false, repacked = false;        // repacked: this warp's slots changed lanes since `mine` was taken
        int wk = PER;                                       // slot indices below wk may be live in this warp
        while (so.M >= 0) {
            // a thread's own maxima of the last pass tell whether it can hold the block's best pair: only those threads look for
            // the tie key (after a rolled-back round `mine` is stale: then every thread looks)
            const bool may_F = force_single || repacked || mine.M == so.M, may_P = force_single || repacked || mine.maxP == so.maxP;
            repacked = false;
            mine.clear();
            if (so.M >= so.maxP) {
                // ------------------------------------------------ merge (a,b) into a: the pair with the largest icf
                int kmine = 0xffff;
                if (may_F)
#pragma unroll
                    for (int k = 0; k < PER; k++) if (k < wk && !(key[k] & CC_GONE) && F[k] == so.M) kmine = min(kmine, (int)(key[k] & 0xffffu));
                const int kF = cc_min_key(kmine, scal + 4, tid, kphase);
                const int a = kF >> 8, b = kF & 0xff;
                for (int t = tid; t < n; t += NT) {
                    int xa = W[a * ns + t], xb = W[b * ns + t];
                    if (t == a || t == b) { xa = 0; xb = 0; }          // rows of inactive nodes are already zero
                    const int nwv = (xa == CC_FORB || xb == CC_FORB) ? CC_FORB : xa + xb;
                    node[t] = make_int4(xa, xb, nwv, 0);
                    W[a * ns + t] = nwv; W[t * ns + a] = nwv; W[b * ns + t] = 0; W[t * ns + b] = 0;
                    if (label[t] == b) label[t] = (uint8_t)a;
                    if (t == b) {                                     // drop b from the list of active nodes
                        active[b] = 0;
                        const int nact = scal[0], pos = apos[b], lastn = alist[nact - 1];
                        alist[pos] = (uint8_t)lastn; apos[lastn] = (uint8_t)pos; scal[0] = nact - 1;
                    }
                }
                __syncthreads();
                // fresh induced costs of the pairs (a,x): G adjacent lanes per x share the third nodes
                {
                    constexpr int G = cc_fresh_g(NT, PER);
                    const int nact = scal[0];
                    const int xi = tid / G, g = tid % G;
                    int x = 0, w = 0;
                    if (xi < nact) { x = alist[xi]; w = node[x].z; }
                    const bool live = w != 0 && w != CC_FORB;
                    int f = 0, p = 0;
                    if (live) {
                        const int32_t* rx = W + x * ns;
                        for (int vi = g; vi < nact; vi += G) {
                            const int v = alist[vi];
                            const int t1 = node[v].z, t2 = rx[v];
                            f += cc_tf(t1, t2); p += cc_tp(t1, t2);
                        }
                    }
#pragma unroll
                    for (int o = G >> 1; o > 0; o >>= 1) { f += __shfl_xor_sync(0xffffffffu, f, o); p += __shfl_xor_sync(0xffffffffu, p, o); }
                    if (live && g == 0) { frF[x] = f + max(w, 0); frP[x] = p + max(-w, 0); }
                }
                __syncthreads();
                // every slot: pairs through a or b take the fresh costs (or die), all others swap the terms through
                // a and b for the term through the merged node
#pragma unroll
                for (int k = 0; k < PER; k++) {
                    if (k >= wk) break;                            // warp-uniform: slots beyond wk are empty since the last packing
                    const uint32_t kq = key[k];
                    if (kq & CC_GONE) continue;
                    const int x = (int)((kq >> 8) & 0xff), y = (int)(kq & 0xff);
                    if (x == a || y == a || x == b || y == b) {
                        // (a,o): continues with the merged weight; (b,o): takes over as (a,o) if a had no edge to o
                        const bool thru_b = x == b || y == b;
                        const int o = thru_b ? (x == b ? y : x) : (x == a ? y : x);
                        const int4 no = node[o];                       // o == a or b: nw = 0 -> the slot of (a,b) dies
                        if (no.z == 0 || no.z == CC_FORB || (thru_b && no.x != 0)) { key[k] = CC_DEAD; continue; }
                        key[k] = (uint32_t)(a < o ? (a << 8) | o : (o << 8) | a) | (no.z > 0 ? CC_POS : 0u);
                        F[k] = frF[o]; P[k] = frP[o];
                    } else {
                        const int4 nx = node[x], ny = node[y];
                        F[k] += cc_tf(nx.z, ny.z) - cc_tf(nx.x, ny.x) - cc_tf(nx.y, ny.y);
                        P[k] += cc_tp(nx.z, ny.z) - cc_tp(nx.x, ny.x) - cc_tp(nx.y, ny.y);
                    }
                    mine.consider(key[k], F[k], P[k]);
                }
                force_single = false;
                const int wlive = __reduce_add_sync(0xffffffffu, mine.live);
                so = cc_reduce<NT>(mine, red, tid, phase);
                // slots only die: once half of a warp's slot rows could be dropped, its survivors are packed row-major
                // into the first rows (lane = j % 32 keeps neighbouring pairs in neighbouring lanes), through this warp's
                // scratch in L2; no other warp is involved
                if (((wlive + 31) >> 5) < wk) {
                    int base = 0;
#pragma unroll
                    for (int k = 0; k < PER; k++) {
                        const bool lv = k < wk && !(key[k] & CC_GONE);
                        const unsigned bal = __ballot_sync(0xffffffffu, lv);
                        if (lv) { const int pos = base + __popc(bal & lt); __stcg(scr + pos, (int)key[k]); __stcg(scr + 32 * PER + pos, F[k]); __stcg(scr + 64 * PER + pos, P[k]); }
                        base += __popc(bal);
                    }
                    __syncwarp();
#pragma unroll
                    for (int k = 0; k < PER; k++) {
                        const int j = k * 32 + lane;
                        if (j < base) { key[k] = (uint32_t)__ldcg(scr + j); F[k] = __ldcg(scr + 32 * PER + j); P[k] = __ldcg(scr + 64 * PER + j); }
                        else key[k] = CC_DEAD;
                    }
                    wk = (base + 31) >> 5;
                    repacked = true;
                    __syncwarp();
                }
            } else if (force_single || so.maxPpos > so.M) {
                // ------------------------------------------------ one sequential forbid: the edge with the largest icp
                int kmine = 0xffff;
                if (may_P)
#pragma unroll
                    for (int k = 0; k < PER; k++) if (k < wk && !(key[k] & CC_GONE) && P[k] == so.maxP) kmine = min(kmine, (int)(key[k] & 0xffffu));
                const int kP = cc_min_key(kmine, scal + 4, tid, kphase);
                const int a = kP >> 8, b = kP & 0xff;
                const int old = W[a * ns + b];                  // set to forbidden after the step's last barrier
#pragma unroll
                for (int k = 0; k < PER; k++) {
                    if (k >= wk) break;                            // warp-uniform: slots beyond wk are empty since the last packing
                    const uint32_t kq = key[k];
                    if (kq & CC_GONE) continue;
                    const int x = (int)((kq >> 8) & 0xff), y = (int)(kq & 0xff);
                    if ((int)(kq & 0xffffu) == kP) { key[k] = CC_DEAD; continue; }
                    int o = -1, third = 0;
                    if (x == a || y == a) { o = x == a ? y : x; third = b; }          // pair (a,o), third node b
                    else if (x == b || y == b) { o = x == b ? y : x; third = a; }     // pair (b,o), third node a
                    if (o >= 0) {
                        const int wt = W[o * ns + third];
                        F[k] -= cc_tf(old, wt); P[k] += cc_tp(CC_FORB, wt) - cc_tp(old, wt);
                    }
                    mine.consider(kq, F[k], P[k]);
                }
                force_single = false;
                so = cc_reduce<NT>(mine, red, tid, phase);
                if (tid == 0) { W[a * ns + b] = CC_FORB; W[b * ns + a] = CC_FORB; }      // read next after the next step's first barrier
            } else {
                // ------------------------------------------------ round: forbid negative candidates with icp > M at once.
                // Forbidding a negative edge changes no icf and only raises icp values, so every such edge stays
                // eligible until it is forbidden: the set forbidden before the next merge is a fixed point that does
                // not depend on the order, PROVIDED no positive edge would be picked in between.  That proviso is
                // checked on the state after the round (max icp over positive candidates <= new max icf); if it
                // fails the round is undone and one sequential step is taken instead.
                const int M = so.M;
                __syncthreads();                               // the masks of the previous round are cleared
                int nfl = 0;
#pragma unroll
                for (int k = 0; k < PER; k++) {
                    if (k >= wk) break;                            // warp-uniform: slots beyond wk are empty since the last packing
                    const uint32_t kq = key[k];
                    if (kq & CC_FLAG) { key[k] = CC_DEAD; continue; }          // forbidden for good in an earlier round
                    if ((kq & (CC_DEAD | CC_POS)) || P[k] <= M) continue;
                    const int x = (int)((kq >> 8) & 0xff), y = (int)(kq & 0xff);
                    key[k] = kq | CC_FLAG; nfl++;
                    atomicOr(&fmask[x * mw + (y >> 5)], 1u << (y & 31)); nodefl[x] = 1;
                    atomicOr(&fmask[y * mw + (x >> 5)], 1u << (x & 31)); nodefl[y] = 1;
                }
                nfl = warp_sum_i32(nfl);
                if (lane == 0 && nfl) atomicAdd(&scal[1], nfl);
                __syncthreads();
                const int nflag = scal[1];
                // D[x][t] = growth of icp(x,t) through the forbidden edges at x: the term through bb grows from
                // min(|w_x,bb|, w_t,bb) to w_t,bb when w_t,bb > 0.  One warp per end node x, lanes over t.
                for (int x = wid; x < n; x += NW) {
                    if (!nodefl[x]) continue;
                    const int32_t* rx = W + x * ns;
                    int g0 = 0, g1 = 0, g2 = 0, g3 = 0, g4 = 0;    // t = lane, lane + 32, ..., lane + 128  (n <= 160)
                    for (int m = 0; m < mw; m++)
                        for (uint32_t bits = fmask[x * mw + m]; bits; bits &= bits - 1) {      // warp-uniform
                            const int bb = m * 32 + __ffs(bits) - 1;
                            const int old = rx[bb];                                           // weight of the forbidden edge < 0
                            const int32_t* rb = W + bb * ns;                                  // w_t,bb = w_bb,t: a row walk
                            if (lane < n) g0 += max(max(rb[lane], 0) + old, 0);
                            if (lane + 32 < n) g1 += max(max(rb[lane + 32], 0) + old, 0);
                            if (lane + 64 < n) g2 += max(max(rb[lane + 64], 0) + old, 0);
                            if (lane + 96 < n) g3 += max(max(rb[lane + 96], 0) + old, 0);
                            if (WIDE5 && lane + 128 < n) g4 += max(max(rb[lane + 128], 0) + old, 0);
                        }
                    int32_t* dx = D + x * ns;
                    if (lane < n) dx[lane] = g0;
                    if (lane + 32 < n) dx[lane + 32] = g1;
                    if (lane + 64 < n) dx[lane + 64] = g2;
                    if (lane + 96 < n) dx[lane + 96] = g3;
                    if (WIDE5 && lane + 128 < n) dx[lane + 128] = g4;
                }
                __syncthreads();
                // the forbidden edges leave (their old weight is parked in D[x][y], which nobody else reads), the icp of
                // the others grows
#pragma unroll
                for (int k = 0; k < PER; k++) {
                    if (k >= wk) break;                            // warp-uniform: slots beyond wk are empty since the last packing
                    const uint32_t kq = key[k];
                    if (kq & CC_DEAD) continue;
                    const int x = (int)((kq >> 8) & 0xff), y = (int)(kq & 0xff);
                    if (kq & CC_FLAG) { D[x * ns + y] = W[x * ns + y]; W[x * ns + y] = CC_FORB; W[y * ns + x] = CC_FORB; continue; }
                    if (nodefl[x]) P[k] += D[x * ns + y];
                    if (nodefl[y]) P[k] += D[y * ns + x];
                    mine.consider(kq, F[k], P[k]);
                }
                const CCBest v = cc_reduce<NT>(mine, red, tid, phase);
                const bool ok = nflag == 1 || v.maxPpos < 0 || v.M < 0 || v.maxPpos <= v.M;
                if (ok) so = v;
                else {
                    // roll back, then one sequential step on the unchanged `so`
                    force_single = true;
#pragma unroll
                    for (int k = 0; k < PER; k++) {
                        if (k >= wk) break;
                        const uint32_t kq = key[k];
                        if (kq & CC_DEAD) continue;
                        const int x = (int)((kq >> 8) & 0xff), y = (int)(kq & 0xff);
                        if (kq & CC_FLAG) { const int w = D[x * ns + y]; W[x * ns + y] = w; W[y * ns + x] = w; key[k] = kq & ~CC_FLAG; continue; }
                        if (nodefl[x]) P[k] -= D[x * ns + y];
                        if (nodefl[y]) P[k] -= D[y * ns + x];
                    }
                    __syncthreads();                           // every thread is done with the masks
                }
                for (int x = tid; x < n; x += NT) if (nodefl[x]) { nodefl[x] = 0; for (int m = 0; m < mw; m++) fmask[x * mw + m] = 0; }
                if (tid == 0) scal[1] = 0;
            }
        }
        // ---- clusters: numbered by smallest member (= representative), ascending
        __syncthreads();
        for (int x = tid; x < n; x += NT) {
            const int rep = label[x];
            int cid = 0;
            for (int y = 0; y < rep; y++) cid += active[y];
            d.fr_cluster[f0 + x] = cid;
        }
        if (tid == 0) d.ch_nclusters[c] = scal[0];
    }
}

}  // namespace ahs
