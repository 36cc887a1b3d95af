// k_thread_canon.cuh — haplotype threading DP for ploidy 5 and 6 on canonical tuples (K4c).
//
// Replaces HaploThreader(p, 32.0, 8.0, false, 0).computePaths (call sites reference src/alignmentstoreadset.cpp:320, :408)
// where the ordered-tuple state space of k_thread — (2p)^p states per column — is out of reach (2.99 M at p = 6).  The
// reference itself fixes p = 2 (:306), so ploidy > 4 has no reference behaviour: the recurrence is rule R3c of
// oracle/core/phase_core.hpp — states are MULTISETS of p local cluster indices (non-decreasing tuples, lexicographic
// rank), a column keeps the first p + 2 entries of covMap, the transition costs 32 per cluster of the multiset
// difference (+ 8 if there is any), ties go to the lowest rank, haplotype labels are threaded greedily afterwards.
//
// min over predecessors without touching all pairs of states:
//   E_j[c] = min { D[s] : s contains the j-multiset c }            down pass over the PREVIOUS column's indices
//   G_j[c] = min { E[c'] + 32 (j - |c'|) : c' inside c }            up pass over THIS column's indices; c' takes part
//                                                                   only if all its clusters exist in the previous column
//   D'[t]  = cost(t) + min( D[s*] for the state s* with the same clusters,  G_p[t] + 8 )
// Both passes walk the levels j of the sub-multiset lattice with precomputed neighbour tables (add one element / delete
// the i-th element); values are (cost, predecessor rank) pairs under lexicographic minimum.  ~30 k table look-ups per
// column at k = 8 instead of 1716^2 = 2.9 M state pairs.
#pragma once
#include "common.cuh"
#include "device_batch.cuh"

namespace ahs {

constexpr int CN_P = 6;                 // largest ploidy
constexpr int CN_K = 8;                 // clusters per column (p + 2 <= 8 = the PosRec capacity)
constexpr int CN_THREADS = 256;

// N(j, k) = number of non-decreasing j-tuples over k symbols = C(k + j - 1, j)
__host__ __device__ inline int cn_count(int j, int k) {
    if (j == 0) return 1;
    if (k <= 0) return 0;
    long long r = 1;
    for (int i = 1; i <= j; i++) r = r * (k - 1 + i) / i;
    return (int)r;
}

// Neighbour tables of the sub-multiset lattice for every alphabet size k = 1..CN_K, levels j = 0..CN_P, in one device
// buffer.  For alphabet k: base[k] = first entry; within it level j starts at lvl[k][j]; entry e of (k, j):
//   tup[e]       the tuple, 4 bits per element (element i at bits 4i)
//   add[e*8+g]   rank within level j+1 of the tuple with g inserted          (j < CN_P, g < k)
//   del[e*6+i]   rank within level j-1 of the tuple without its element i    (j >= 1, i < j)
struct CanonTables {
    int32_t base[CN_K + 1];
    int32_t lvl[CN_K + 1][CN_P + 2];
    const uint32_t* tup; const uint16_t* add; const uint16_t* del;
    int32_t nn[CN_P + 1][CN_K + 1];          // cn_count(j, k)
};

// lexicographic rank of a non-decreasing tuple x[0..j) over k symbols
__host__ __device__ inline int cn_rank(const uint8_t* x, int j, int k, const int32_t (*nn)[CN_K + 1]) {
    int r = 0, prev = 0;
    for (int i = 0; i < j; i++) { for (int v = prev; v < x[i]; v++) r += nn[j - 1 - i][k - v]; prev = x[i]; }
    return r;
}

struct CNVA { int v; int a; };          // (cost, predecessor rank), lexicographic minimum
__device__ __forceinline__ void cn_min(CNVA& x, int v, int a) { if (v < x.v || (v == x.v && a < x.a)) { x.v = v; x.a = a; } }

__host__ __device__ inline size_t cn_smem_bytes() {
    const size_t T = 3003;                                   // entries of alphabet 8: C(14, 6)
    return T * (4 + 2) * 2 + 1716 * 4 + 1716 + 2 * sizeof(PosRec) + 256;
}

// GT: caller genotypes (d.gt_col) are present.  Two instances, so that the plain one is the kernel without any genotype code
// (48 registers).  The GT instance declares 3 blocks per SM — what the 64 KB of shared memory of a block allows anyway —
// because ptxas otherwise keeps it at 48 registers and spills; with the hint it takes 56 and spills nothing.
template <bool GT>
__global__ void __launch_bounds__(CN_THREADS, GT ? 3 : 0) k_thread_canon(DB d, CanonTables tb, int32_t* __restrict__ work_counter) {
    extern __shared__ __align__(16) unsigned char cn_sm[];
    const int p = d.ploidy;
    int32_t* Ev = (int32_t*)cn_sm; int32_t* Gv = Ev + 3003; int32_t* Dcur = Gv + 3003;
    uint16_t* Ea = (uint16_t*)(Dcur + 1716); uint16_t* Ga = Ea + 3004;
    int8_t* cc = (int8_t*)(Ga + 3004);
    PosRec* s_rec = (PosRec*)(((uintptr_t)(cc + 1716) + 15) & ~(uintptr_t)15);
    int* s_misc = (int*)(s_rec + 2);                         // [0] chain, [1] any conform, [8..16) cur -> prev local index
    const int tid = threadIdx.x, nt = blockDim.x;
    while (true) {
        if (tid == 0) s_misc[0] = atomicAdd(work_counter, 1);
        __syncthreads();
        const int c = s_misc[0];
        __syncthreads();
        if (c >= d.C) break;
        if (d.ch_status[c] != AHS_CHAIN_OK) continue;
        const int64_t p0 = d.pos_off[c];
        const int n_pos = (int)(d.pos_off[c + 1] - p0);
        if (n_pos == 0) continue;
        uint16_t* back = d.back + d.back_off[c];
        const int SM = d.S_max;
        int kp = 0;
        for (int q = 0; q < n_pos; q++) {
            if (tid == 0) s_rec[q & 1] = d.rec[p0 + q];
            if (tid == 0) s_misc[1] = 0;
            __syncthreads();
            const PosRec& R = s_rec[q & 1];
            const PosRec& Rp = s_rec[(q & 1) ^ 1];
            const int kc = R.k;
            const int bc = tb.base[kc], S = tb.nn[p][kc];
            const uint32_t* tupc = tb.tup + bc;
            // ---- per-state genotype conformity and coverage cost (rule R3; they depend on the multiset only)
            int any = 0;
            for (int t = tid; t < S; t += nt) {
                const uint32_t tp = tupc[tb.lvl[kc][p] + t];
                int dig[CN_P];
#pragma unroll
                for (int h = 0; h < CN_P; h++) dig[h] = (int)((tp >> (4 * h)) & 15u);
                bool conform = false;
                for (int h = 1; h < p; h++) conform |= R.cons_asc[dig[h]] != R.cons_asc[dig[0]];
                int cost = 0;
                for (int h = 0; h < p; h++) {
                    int m = 0; for (int g = 0; g < p; g++) m += dig[g] == dig[h];
                    const uint64_t lhs = (uint64_t)R.cnt_asc[dig[h]] * (uint64_t)(2 * p);
                    if (lhs < (uint64_t)(2 * m - 1) * R.total || lhs > (uint64_t)(2 * m + 1) * R.total) cost++;
                }
                cc[t] = conform ? (int8_t)cost : (int8_t)(-1 - cost);
                any |= conform;
            }
            // caller genotype known at this column (ahs_phase_batch_genotyped): conformity is instead the multiset test of its
            // key (genotype_key); every thread re-marks the states it has just written
            if (GT) {
                const uint64_t G = d.gt_col[p0 + q];
                if (G) {
                    any = 0;
                    for (int t = tid; t < S; t += nt) {
                        const uint32_t tp = tupc[tb.lvl[kc][p] + t];
                        uint64_t key = 0;
                        for (int h = 0; h < p; h++) key += 1ull << (4 * R.cons_asc[(tp >> (4 * h)) & 15u]);
                        const int v = cc[t], cost = v >= 0 ? v : -1 - v;
                        cc[t] = key == G ? (int8_t)cost : (int8_t)(-1 - cost);
                        any |= key == G;
                    }
                }
            }
            any = __syncthreads_or(any);
            if (q == 0) {
                for (int t = tid; t < S; t += nt) { const int v = cc[t]; Dcur[t] = (v >= 0) ? v : (any ? DP_INF : (-1 - v)); }
            } else {
                const int bp = tb.base[kp], Sp = tb.nn[p][kp];
                const int32_t* lvp = tb.lvl[kp]; const int32_t* lvc = tb.lvl[kc];
                // this column's local index -> the previous column's local index of the same cluster
                if (tid < CN_K) { int m = -1; if (tid < kc) for (int x = 0; x < kp; x++) if (Rp.gid[x] == R.gid[tid]) { m = x; break; } s_misc[8 + tid] = m; }
                // level p of E = the previous column (kept in Dcur)
                for (int s = tid; s < Sp; s += nt) { Ev[lvp[p] + s] = Dcur[s]; Ea[lvp[p] + s] = (uint16_t)s; }
                __syncthreads();
                // ---- down pass: E_j[c] = min over the inserted element g of E_{j+1}[c + g]
                for (int j = p - 1; j >= 0; j--) {
                    const int cnt = tb.nn[j][kp];
                    for (int e = tid; e < cnt; e += nt) {
                        const uint16_t* ad = tb.add + (size_t)(bp + lvp[j] + e) * 8;
                        CNVA b{INT32_MAX, INT32_MAX};
                        for (int g = 0; g < kp; g++) { const int u = lvp[j + 1] + ad[g]; cn_min(b, Ev[u], Ea[u]); }
                        Ev[lvp[j] + e] = b.v; Ea[lvp[j] + e] = (uint16_t)b.a;
                    }
                    __syncthreads();
                }
                // ---- up pass: G_j[c] = min(E_j[c mapped to the previous column], min over the deleted element of G_{j-1} + 32)
                if (tid == 0) { Gv[lvc[0]] = Ev[lvp[0]]; Ga[lvc[0]] = Ea[lvp[0]]; }
                __syncthreads();
                for (int j = 1; j <= p; j++) {
                    const int cnt = tb.nn[j][kc];
                    for (int e = tid; e < cnt; e += nt) {
                        const uint32_t tp = tupc[lvc[j] + e];
                        CNVA b{INT32_MAX, INT32_MAX};
                        // the multiset itself, if all its clusters exist in the previous column
                        {
                            uint8_t x[CN_P]; bool ok = true;
                            for (int i = 0; i < j; i++) { const int m = s_misc[8 + ((tp >> (4 * i)) & 15u)]; if (m < 0) { ok = false; break; } x[i] = (uint8_t)m; }
                            if (ok) {
                                for (int i = 1; i < j; i++) { const uint8_t v = x[i]; int y = i - 1; while (y >= 0 && x[y] > v) { x[y + 1] = x[y]; y--; } x[y + 1] = v; }
                                const int u = lvp[j] + cn_rank(x, j, kp, tb.nn);
                                if (Ev[u] < DP_INF) cn_min(b, Ev[u], Ea[u]);
                            }
                        }
                        const uint16_t* dl = tb.del + (size_t)(bc + lvc[j] + e) * 6;
                        for (int i = 0; i < j; i++) {
                            if (i > 0 && ((tp >> (4 * i)) & 15u) == ((tp >> (4 * (i - 1))) & 15u)) continue;
                            const int u = lvc[j - 1] + dl[i];
                            if (Gv[u] < DP_INF) cn_min(b, Gv[u] + 32, Ga[u]);
                        }
                        Gv[lvc[j] + e] = b.v == INT32_MAX ? DP_INF : b.v; Ga[lvc[j] + e] = (uint16_t)(b.a == INT32_MAX ? 0 : b.a);
                    }
                    __syncthreads();
                }
                // ---- this column: any switch (+8) against the predecessor with the same clusters
                for (int t = tid; t < S; t += nt) {
                    const int u = lvc[p] + t;
                    CNVA b{INT32_MAX, INT32_MAX};
                    if (Gv[u] < DP_INF) cn_min(b, Gv[u] + 8, Ga[u]);
                    {
                        const uint32_t tp = tupc[u];
                        uint8_t x[CN_P]; bool ok = true;
                        for (int i = 0; i < p; i++) { const int m = s_misc[8 + ((tp >> (4 * i)) & 15u)]; if (m < 0) { ok = false; break; } x[i] = (uint8_t)m; }
                        if (ok) {
                            for (int i = 1; i < p; i++) { const uint8_t v = x[i]; int y = i - 1; while (y >= 0 && x[y] > v) { x[y + 1] = x[y]; y--; } x[y + 1] = v; }
                            const int s = cn_rank(x, p, kp, tb.nn);
                            const int dv = Ev[lvp[p] + s];
                            if (dv < DP_INF) cn_min(b, dv, s);
                        }
                    }
                    const int v = cc[t];
                    const bool allowed = (v >= 0) || !any;
                    const int cost = v >= 0 ? v : (-1 - v);
                    cc[t] = 0;
                    // Dcur is still the previous column for the threads that have not got here: write after the barrier
                    Gv[u] = (allowed && b.v != INT32_MAX) ? min(b.v + cost, DP_INF) : DP_INF;
                    back[(int64_t)q * SM + t] = (uint16_t)(b.a == INT32_MAX ? 0 : b.a);
                }
                __syncthreads();
                for (int t = tid; t < S; t += nt) Dcur[t] = Gv[lvc[p] + t];
            }
            __syncthreads();
            kp = kc;
        }
        // ---- final minimum (lowest rank), backtrace, haplotype labels threaded forward (rule R3c)
        if (tid == 0) {
            const int S = tb.nn[p][kp];
            int best = INT32_MAX, cur = 0;
            for (int t = 0; t < S; t++) if (Dcur[t] < best) { best = Dcur[t]; cur = t; }
            d.dp_cost[c] = (double)best;
            for (int q = n_pos - 1; q >= 0; q--) { d.path[(p0 + q) * p] = cur; if (q > 0) cur = back[(int64_t)q * SM + cur]; }      // state per position, parked in path
            int prev[CN_P];
            for (int q = 0; q < n_pos; q++) {
                const PosRec& R = d.rec[p0 + q];
                const int kc = R.k;
                const uint32_t tp = tb.tup[tb.base[kc] + tb.lvl[kc][p] + d.path[(p0 + q) * p]];
                int el[CN_P], now[CN_P]; bool claimed[CN_P], placed[CN_P];
                for (int h = 0; h < p; h++) { el[h] = (int)((tp >> (4 * h)) & 15u); claimed[h] = false; placed[h] = false; }
                if (q == 0) { for (int h = 0; h < p; h++) now[h] = R.gid[el[h]]; }
                else {
                    for (int h = 0; h < p; h++)
                        for (int e = 0; e < p; e++) if (!claimed[e] && R.gid[el[e]] == prev[h]) { claimed[e] = true; placed[h] = true; now[h] = prev[h]; break; }
                    int e = 0;
                    for (int h = 0; h < p; h++) if (!placed[h]) { while (claimed[e]) e++; now[h] = R.gid[el[e]]; claimed[e] = true; }
                }
                for (int h = 0; h < p; h++) {
                    prev[h] = now[h];
                    d.path[(p0 + q) * p + h] = now[h];
                    int l = 0; for (int x = 0; x < kc; x++) if (R.gid[x] == now[h]) l = x;
                    d.hap_allele[(p0 + q) * p + h] = R.cons_cm[l];
                }
            }
        }
        __syncthreads();
    }
}

}  // namespace ahs
