// k_thread.cuh — per-position cluster coverage / consensus (K3), haplotype threading DP (K4) and
// the CSR result writers.
//
// K3 replaces get_coverage (:660-697), get_pos_to_clusters_map (:751-779),
// get_local_cluster_consensus / get_single_cluster_consensus_frac (:550-655) and the re-packing at
// :378-404 of reference src/alignmentstoreadset.cpp — including the fact that the coverage and
// consensus vectors handed to the threader are in ascending-cluster-id order while covMap is in
// descending-coverage order (SURVEY A#12).  Coverage is kept as (count, total): every comparison
// the reference makes on count/total doubles is decided identically by the integer cross product.
//
// K4 replaces HaploThreader(2,32.0,8.0,false,0).computePaths (:320,:408; algorithm:
// oracle/core/phase_core.hpp rule R3).  The transition cost 32*(#switched haplotypes) is separable
// over haplotypes, so the min over predecessors is taken one tuple coordinate at a time (least
// significant first, ties -> smallest predecessor digit), which yields exactly the minimum and
// the lowest-code argmin of the all-pairs definition; the affine 8 is applied afterwards against
// the unique zero-switch predecessor.  Costs are integers.
#pragma once
#include "common.cuh"
#include "device_batch.cuh"
#include "k_project.cuh"

namespace ahs {

constexpr int K3_CAP = 128;      // clusters per position held in shared memory (k_consensus)
constexpr int K3C_CAP = 16;      // clusters per chain handled by the warp-per-chain kernel (k_consensus_chain)
constexpr int K3C_READS = 128;   // ... and final reads per chain (a lane walks all of them; longer chains go position-parallel)

template <int BITS, int G>
__global__ void __launch_bounds__(128) k_consensus(DB d) {
    constexpr int NG = 128 / G;                                       // position groups per block
    __shared__ int32_t s_id[NG][K3_CAP], s_cnt[NG][K3_CAP], s_key[NG][K3_CAP], s_idx[NG][K3_CAP];
    __shared__ uint8_t s_cons[NG][K3_CAP];
    const unsigned gm = grp_mask<G>();
    const int gl = lane_id() % G, wib = threadIdx.x / G;
    const int p = d.ploidy;
    for (int64_t gp = blockIdx.x * (int64_t)NG + wib; gp < d.NP; gp += (int64_t)gridDim.x * NG) {
        const int c = d.pos_chain[gp];
        if (BITS == 2 && d.ch_nclusters[c] <= K3C_CAP && d.frow_off[c + 1] - d.frow_off[c] <= K3C_READS) continue;      // done by k_consensus_chain
        const int b = d.pos[gp];
        const int64_t f0 = d.frow_off[c];
        const int n_c = (int)(d.frow_off[c + 1] - f0);
        const int32_t* first = d.fr_first + f0; const int32_t* lastp = d.fr_last + f0; const int32_t* cl = d.fr_cluster + f0;
        const int words = d.ch_words[c];
        const uint32_t* rows = d.codes + d.code_off[c];
        const int64_t gb = d.bubble_off[c] + b;
        const int K = (int)(d.allele_off[gb + 1] - d.allele_off[gb]);
        // candidate band: first <= b and first >= b - maxspan
        int lo, hi;
        { int x = -1, y = n_c; while (x + 1 < y) { int m = (x + y) >> 1; if (first[m] <= b) x = m; else y = m; } hi = x;
          const int bound = b - d.ch_maxspan[c]; x = -1; y = n_c; while (x + 1 < y) { int m = (x + y) >> 1; if (first[m] >= bound) y = m; else x = m; } lo = y; }
        int cur = -1, ncl = 0; uint32_t total = 0; bool overflow = false;
        while (true) {
            int nxt = INT32_MAX;
            for (int i = lo + gl; i <= hi; i += G)
                if (lastp[i] >= b && cl[i] > cur && get_code(rows + (int64_t)i * words, b, BITS)) nxt = min(nxt, cl[i]);
            nxt = __reduce_min_sync(gm, nxt);
            if (nxt == INT32_MAX) break;
            constexpr int NA_MAX = BITS == 2 ? 3 : MAX_ALLELES;       // 2-bit codes hold at most 3 alleles
            uint32_t ac[NA_MAX];
#pragma unroll
            for (int a = 0; a < NA_MAX; a++) ac[a] = 0;
            for (int i = lo + gl; i <= hi; i += G)
                if (lastp[i] >= b && cl[i] == nxt) {
                    const uint32_t code = get_code(rows + (int64_t)i * words, b, BITS);
#pragma unroll
                    for (int a = 0; a < NA_MAX; a++) ac[a] += (code == (uint32_t)(a + 1)) ? 1u : 0u;
                }
            uint32_t cnt = 0, best = 0; int cons = 0;
#pragma unroll
            for (int a = 0; a < NA_MAX; a++) if (a < K) {
                const uint32_t v = (uint32_t)__reduce_add_sync(gm, (int)ac[a]);
                cnt += v;
                if (v > best) { best = v; cons = a; }               // ties -> smallest allele (:633-649, A#13)
            }
            if (ncl < K3_CAP) { if (gl == 0) { s_id[wib][ncl] = nxt; s_cnt[wib][ncl] = (int32_t)cnt; s_cons[wib][ncl] = (uint8_t)cons; } }
            else overflow = true;
            ncl++; total += cnt; cur = nxt;
        }
        __syncwarp(gm);
        if (overflow) { if (gl == 0) atomicMax(&d.ch_status[c], AHS_CHAIN_TOO_LARGE); continue; }
        if (gl == 0) {
            PosRec r;
            r.total = total; r.pad[0] = r.pad[1] = r.pad[2] = 0;
            for (int x = 0; x < ncl; x++) { s_key[wib][x] = s_cnt[wib][x]; s_idx[wib][x] = x; }
            KV kv; kv.k = s_key[wib]; kv.v = s_idx[wib];
            kv_std_sort<true>(kv, ncl);                            // std::sort(A, cmp) on coverage, descending (:720)
            int k = min(ncl, 2 * p);
            for (int i = p; i < min(ncl, 2 * p); i++)
                if ((uint64_t)s_cnt[wib][s_idx[wib][i]] * (uint64_t)(8 * p) < (uint64_t)total) { k = i; break; }   // cov < 1/(8p), :768
            // the DP column: all of covMap[pos] up to ploidy 4, its first p + 2 entries above (rule R3c); the consensus list
            // is the one of ALL covMap clusters in ascending id order (A#12), of which the column reads the first r.k entries
            const int kr = p > 4 ? min(k, p + 2) : k;
            r.k = (uint8_t)kr;
            int sel[MAX_K];
            for (int l = 0; l < PR_K; l++) { r.gid[l] = -1; r.cnt_asc[l] = 0; r.cons_asc[l] = 0; r.cons_cm[l] = 0; }
            for (int l = 0; l < k; l++) sel[l] = s_idx[wib][l];
            for (int l = 0; l < kr; l++) { r.gid[l] = s_id[wib][sel[l]]; r.cons_cm[l] = s_cons[wib][sel[l]]; r.cnt_asc[l] = (uint32_t)s_cnt[wib][l]; }
            for (int x = 1; x < k; x++) { int v = sel[x], y = x - 1; while (y >= 0 && sel[y] > v) { sel[y + 1] = sel[y]; y--; } sel[y + 1] = v; }
            for (int l = 0; l < kr; l++) r.cons_asc[l] = s_cons[wib][sel[l]];
            d.rec[gp] = r;
        }
        __syncwarp(gm);
    }
}

// ---------------------------------------------------------------- K3, common case: one warp per chain
// 2-bit codes (<= 3 alleles) and at most K3C_CAP clusters in the chain: one lane per covered position walks the
// chain's reads once and counts (cluster, allele) in a small shared-memory table; the selection of covMap, the
// consensus and the re-packing are the same statements as in k_consensus, executed by 32 positions at a time.
__global__ void __launch_bounds__(128) k_consensus_chain(DB d) {
    __shared__ uint16_t s_cnt[4][32][K3C_CAP][3];                      // [warp][position lane][cluster][allele]
    __shared__ int32_t s_key[4][32][K3C_CAP], s_idx[4][32][K3C_CAP];
    const int lane = lane_id(), wib = threadIdx.x >> 5;
    const int p = d.ploidy;
    for (int c = blockIdx.x * 4 + wib; c < d.C; c += gridDim.x * 4) {
        if (d.ch_status[c] != AHS_CHAIN_OK) continue;
        const int ncl = d.ch_nclusters[c];
        const int64_t f0 = d.frow_off[c], p0 = d.pos_off[c];
        const int n_c = (int)(d.frow_off[c + 1] - f0), n_pos = (int)(d.pos_off[c + 1] - p0);
        if (ncl > K3C_CAP || n_c > K3C_READS) continue;                // k_consensus takes this chain
        const int32_t* first = d.fr_first + f0; const int32_t* lastp = d.fr_last + f0; const int32_t* cl = d.fr_cluster + f0;
        const int words = d.ch_words[c];
        const uint32_t* rows = d.codes + d.code_off[c];
        for (int q0 = 0; q0 < n_pos; q0 += 32) {
            const int q = q0 + lane;
            const bool live = q < n_pos;
            const int b = live ? d.pos[p0 + q] : -1;
            uint16_t (*cnt)[3] = s_cnt[wib][lane];
            for (int k = 0; k < ncl; k++) { cnt[k][0] = 0; cnt[k][1] = 0; cnt[k][2] = 0; }
            if (live) for (int i = 0; i < n_c; i++) {
                if (first[i] > b) break;                                // reads are sorted by first position
                if (lastp[i] < b) continue;
                const uint32_t code = get_code(rows + (int64_t)i * words, b, 2);
                if (code) cnt[cl[i]][code - 1]++;
            }
            if (live) {
                const int64_t gb = d.bubble_off[c] + b;
                const int K = (int)(d.allele_off[gb + 1] - d.allele_off[gb]);
                // clusters present at this position, ascending id (= the order k_consensus discovers them in)
                int32_t* key = s_key[wib][lane]; int32_t* idx = s_idx[wib][lane];
                int ids[K3C_CAP]; uint8_t cons[K3C_CAP]; int cn[K3C_CAP];
                int m = 0; uint32_t total = 0;
#pragma unroll
                for (int k = 0; k < K3C_CAP; k++) if (k < ncl) {
                    uint32_t tot = 0, best = 0; int best_a = 0;
                    for (int a = 0; a < 3; a++) if (a < K) { const uint32_t v = cnt[k][a]; tot += v; if (v > best) { best = v; best_a = a; } }   // ties -> smallest allele
                    if (tot > 0) { ids[m] = k; cn[m] = (int)tot; cons[m] = (uint8_t)best_a; key[m] = (int)tot; idx[m] = m; m++; total += tot; }
                }
                PosRec r;
                r.total = total; r.pad[0] = r.pad[1] = r.pad[2] = 0;
                KV kv; kv.k = key; kv.v = idx;
                kv_std_sort<true>(kv, m);                              // std::sort(A, cmp) on coverage, descending (:720)
                int k = min(m, 2 * p);
                for (int i = p; i < min(m, 2 * p); i++)
                    if ((uint64_t)cn[idx[i]] * (uint64_t)(8 * p) < (uint64_t)total) { k = i; break; }          // cov < 1/(8p), :768
                const int kr = p > 4 ? min(k, p + 2) : k;             // see k_consensus
                r.k = (uint8_t)kr;
                int sel[MAX_K];
                for (int l = 0; l < PR_K; l++) { r.gid[l] = -1; r.cnt_asc[l] = 0; r.cons_asc[l] = 0; r.cons_cm[l] = 0; }
                for (int l = 0; l < k; l++) sel[l] = idx[l];
                for (int l = 0; l < kr; l++) { r.gid[l] = ids[sel[l]]; r.cons_cm[l] = cons[sel[l]]; r.cnt_asc[l] = (uint32_t)cn[l]; }
                for (int x = 1; x < k; x++) { int v = sel[x], y = x - 1; while (y >= 0 && sel[y] > v) { sel[y + 1] = sel[y]; y--; } sel[y + 1] = v; }
                for (int l = 0; l < kr; l++) r.cons_asc[l] = cons[sel[l]];
                d.rec[p0 + q] = r;
            }
            __syncwarp();
        }
    }
}

// ---------------------------------------------------------------- K4: threading DP, one block per chain
constexpr int DP_THREADS = 128;

__device__ __forceinline__ int ipow(int b, int e) { int r = 1; for (int i = 0; i < e; i++) r *= b; return r; }

// caller genotypes (ahs_phase_batch_genotyped): the key of every DP column, from the dosages of its bubble (0 = unknown).
// The dosages were validated by k_validate.
__global__ void k_gt_columns(DB d) {
    for (int64_t gp = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; gp < d.NP; gp += (int64_t)gridDim.x * blockDim.x) {
        const int64_t gb = d.bubble_off[d.pos_chain[gp]] + d.pos[gp];
        int sum;
        d.gt_col[gp] = genotype_key(d.allele_dosage + d.allele_off[gb], (int)(d.allele_off[gb + 1] - d.allele_off[gb]), sum);
    }
}

__global__ void __launch_bounds__(DP_THREADS) k_thread(DB d, int32_t* __restrict__ work_counter) {
    extern __shared__ int32_t smem[];
    const int SM = d.S_max, p = d.ploidy;
    int32_t* Dprev = smem; int32_t* Dcur = smem + SM; int32_t* Xa = smem + 2 * SM; int32_t* Xb = smem + 3 * SM;
    uint16_t* Aa = (uint16_t*)(smem + 4 * SM); uint16_t* Ab = Aa + SM;
    int8_t* cc = (int8_t*)(Ab + SM);                    // covcost, -1 = not genotype conform
    __shared__ PosRec s_rec[2];
    __shared__ int s_chain;
    __shared__ uint64_t s_gt;                           // genotype key of the column (caller genotypes only)
    const int tid = threadIdx.x, nt = blockDim.x;
    while (true) {
        if (tid == 0) s_chain = atomicAdd(work_counter, 1);
        __syncthreads();
        const int c = s_chain;
        __syncthreads();
        if (c >= d.C) break;
        if (d.ch_status[c] != AHS_CHAIN_OK) continue;
        const int64_t p0 = d.pos_off[c];
        const int n_pos = (int)(d.pos_off[c + 1] - p0);
        if (n_pos == 0) continue;
        uint16_t* back = d.back + d.back_off[c];
        int kp = 0;
        for (int q = 0; q < n_pos; q++) {
            if (tid == 0) { s_rec[q & 1] = d.rec[p0 + q]; if (d.gt_col) s_gt = d.gt_col[p0 + q]; }
            __syncthreads();
            const PosRec& R = s_rec[q & 1];
            const PosRec& Rp = s_rec[(q & 1) ^ 1];
            const int kc = R.k;
            const int S = ipow(kc, p);
            // ---- per-tuple genotype conformity and coverage cost
            int any = 0;
            for (int t = tid; t < S; t += nt) {
                int dig[MAX_PLOIDY]; { int x = t; for (int h = p - 1; h >= 0; h--) { dig[h] = x % kc; x /= kc; } }
                bool conform;
                const uint64_t G = d.gt_col ? s_gt : 0; // 0: the built-in genotype rule
                if (G) { uint64_t key = 0; for (int h = 0; h < p; h++) key += 1ull << (4 * R.cons_asc[dig[h]]); conform = key == G; }
                else if (p == 2) { const int a0 = R.cons_asc[dig[0]], a1 = R.cons_asc[dig[1]]; conform = (a0 == 0 && a1 == 1) || (a0 == 1 && a1 == 0); }
                else { conform = false; for (int h = 1; h < p; h++) conform |= R.cons_asc[dig[h]] != R.cons_asc[dig[0]]; }
                int cost = 0;
                for (int h = 0; h < p; h++) {
                    int m = 0; for (int g = 0; g < p; g++) m += dig[g] == dig[h];
                    const uint64_t lhs = (uint64_t)R.cnt_asc[dig[h]] * (uint64_t)(2 * p);
                    if (lhs < (uint64_t)(2 * m - 1) * R.total || lhs > (uint64_t)(2 * m + 1) * R.total) cost++;
                }
                cc[t] = conform ? (int8_t)cost : (int8_t)(-1 - cost);
                any |= conform;
            }
            any = __syncthreads_or(any);
            if (q == 0) {
                for (int t = tid; t < S; t += nt) { const int v = cc[t]; Dcur[t] = (v >= 0) ? v : (any ? DP_INF : (-1 - v)); }
            } else {
                // ---- factorised min over predecessors
                const int Sp = ipow(kp, p);
                for (int t = tid; t < Sp; t += nt) { Xa[t] = Dprev[t]; Aa[t] = 0; }
                __syncthreads();
                int32_t* Xin = Xa; int32_t* Xout = Xb; uint16_t* Ain = Aa; uint16_t* Aout = Ab;
                for (int h = p - 1; h >= 0; h--) {
                    const int lowsz = ipow(kc, p - 1 - h), highsz = ipow(kp, h), wpred = ipow(kp, p - 1 - h);
                    const int n_out = highsz * kc * lowsz;
                    for (int o = tid; o < n_out; o += nt) {
                        const int low = o % lowsz, rest = o / lowsz, th = rest % kc, high = rest / kc;
                        const int gcur = R.gid[th];
                        int best = INT32_MAX, barg = 0;
                        for (int sh = 0; sh < kp; sh++) {
                            const int in = (high * kp + sh) * lowsz + low;
                            const int v = Xin[in] + (Rp.gid[sh] != gcur ? 32 : 0);
                            if (v < best) { best = v; barg = Ain[in] + sh * wpred; }
                        }
                        Xout[o] = best; Aout[o] = (uint16_t)barg;
                    }
                    __syncthreads();
                    int32_t* tx = Xin; Xin = Xout; Xout = tx; uint16_t* ta = Ain; Ain = Aout; Aout = ta;
                }
                // ---- affine part and zero-switch predecessor
                for (int t = tid; t < S; t += nt) {
                    int dig[MAX_PLOIDY]; { int x = t; for (int h = p - 1; h >= 0; h--) { dig[h] = x % kc; x /= kc; } }
                    int val = Xin[t]; int pred = Ain[t];
                    int sw = 0; { int x = pred; for (int h = p - 1; h >= 0; h--) { const int sh = x % kp; x /= kp; sw += Rp.gid[sh] != R.gid[dig[h]]; } }
                    if (sw) {
                        val += 8;
                        int sstar = 0; bool ok = true;
                        for (int h = 0; h < p; h++) {
                            int l = -1; for (int x = 0; x < kp; x++) if (Rp.gid[x] == R.gid[dig[h]]) l = x;
                            if (l < 0) { ok = false; break; }
                            sstar = sstar * kp + l;
                        }
                        if (ok) { const int v2 = Dprev[sstar]; if (v2 < val || (v2 == val && sstar < pred)) { val = v2; pred = sstar; } }
                    }
                    const int v = cc[t];
                    const bool allowed = (v >= 0) || !any;
                    const int cost = v >= 0 ? v : (-1 - v);
                    Dcur[t] = allowed ? min(val + cost, DP_INF) : DP_INF;
                    back[(int64_t)q * SM + t] = (uint16_t)pred;
                }
            }
            __syncthreads();
            { int32_t* tx = Dprev; Dprev = Dcur; Dcur = tx; }
            kp = kc;
        }
        // ---- final minimum (lowest code) and backtrace
        if (tid == 0) {
            const int S = ipow(kp, p);
            int best = INT32_MAX, cur = 0;
            for (int t = 0; t < S; t++) if (Dprev[t] < best) { best = Dprev[t]; cur = t; }
            d.dp_cost[c] = (double)best;
            for (int q = n_pos - 1; q >= 0; q--) {
                const PosRec& R = d.rec[p0 + q];
                const int kc = R.k;
                int x = cur;
                for (int h = p - 1; h >= 0; h--) {
                    const int dg = x % kc; x /= kc;
                    d.path[(p0 + q) * p + h] = R.gid[dg];
                    d.hap_allele[(p0 + q) * p + h] = R.cons_cm[dg];
                }
                if (q > 0) cur = back[(int64_t)q * SM + cur];
            }
        }
        __syncthreads();
    }
}

// ---------------------------------------------------------------- K4 for ploidy 2: one WARP per chain
// At ploidy 2 a column has at most 4 x 4 = 16 states, so a warp holds the whole DP column in registers (lane = state
// code), the per-position record (22 words) arrives as one coalesced load that is prefetched one position ahead, the
// min over predecessors is 16 shuffles, and there is no block barrier.  Same recurrence, same tie rules (lowest
// predecessor code, lowest final code) as k_thread / rule R3.
static_assert(sizeof(PosRec) == 88, "k_thread2 reads PosRec as 22 words");

__global__ void __launch_bounds__(256) k_thread2(DB d, int32_t* __restrict__ work_counter) {
    const int lane = lane_id();
    const unsigned full = 0xffffffffu;
    while (true) {
        int c = 0;
        if (lane == 0) c = atomicAdd(work_counter, 1);
        c = __shfl_sync(full, c, 0);
        if (c >= d.C) break;
        if (d.ch_status[c] != AHS_CHAIN_OK) continue;
        const int64_t p0 = d.pos_off[c];
        const int n_pos = (int)(d.pos_off[c + 1] - p0);
        if (n_pos == 0) continue;
        uint16_t* back = d.back + d.back_off[c];                       // 16 predecessor codes per position
        const uint32_t* recw = (const uint32_t*)(d.rec + p0);
        // caller genotypes: lanes 22 and 23 carry the column's key (low, high word) next to the record
        const uint32_t* gtw = d.gt_col ? (const uint32_t*)(d.gt_col + p0) : nullptr;
        uint32_t rw = lane < 22 ? recw[lane] : (gtw && lane < 24) ? gtw[lane - 22] : 0u;
        int Dprev = DP_INF, gp0 = -1, gp1 = -1, kp = 0;
        for (int q = 0; q < n_pos; q++) {
            uint32_t rw_next = (q + 1 < n_pos && lane < 22) ? recw[(int64_t)(q + 1) * 22 + lane] : 0u;
            if (gtw && q + 1 < n_pos && (lane == 22 || lane == 23)) rw_next = gtw[(int64_t)(q + 1) * 2 + lane - 22];
            const uint32_t total = __shfl_sync(full, rw, 0);
            const int kc = (int)(__shfl_sync(full, rw, 1) & 0xffu);
            const int S = kc * kc;
            const bool valid = lane < S;
            const int d0 = valid ? lane / kc : 0, d1 = valid ? lane % kc : 0;       // haplotype 0 = most significant digit
            const int g0 = (int)__shfl_sync(full, rw, 2 + d0), g1 = (int)__shfl_sync(full, rw, 2 + d1);
            const uint32_t c0 = __shfl_sync(full, rw, 10 + d0), c1 = __shfl_sync(full, rw, 10 + d1);
            const int a0 = (int)((__shfl_sync(full, rw, 18 + (d0 >> 2)) >> (8 * (d0 & 3))) & 0xffu);
            const int a1 = (int)((__shfl_sync(full, rw, 18 + (d1 >> 2)) >> (8 * (d1 & 3))) & 0xffu);
            bool conform;
            if (gtw) {                                                 // key == (G ? G : 0x11): {0:1, 1:1} where the genotype is unknown
                const uint64_t G = ((uint64_t)__shfl_sync(full, rw, 23) << 32) | __shfl_sync(full, rw, 22);
                conform = (1ull << (4 * a0)) + (1ull << (4 * a1)) == (G ? G : 0x11ull);
            } else conform = (a0 == 0 && a1 == 1) || (a0 == 1 && a1 == 0);
            const uint64_t m = d0 == d1 ? 2 : 1;
            int cost = 0;
            { const uint64_t lhs = (uint64_t)c0 * 4; if (lhs < (2 * m - 1) * total || lhs > (2 * m + 1) * total) cost++; }
            { const uint64_t lhs = (uint64_t)c1 * 4; if (lhs < (2 * m - 1) * total || lhs > (2 * m + 1) * total) cost++; }
            const bool any = __any_sync(full, valid && conform);
            const bool allowed = conform || !any;
            int Dcur;
            if (q == 0) Dcur = allowed ? cost : DP_INF;
            else {
                int best = INT32_MAX, arg = 0;
                const int Sp = kp * kp;
                for (int sidx = 0; sidx < Sp; sidx++) {
                    const int dv = __shfl_sync(full, Dprev, sidx);
                    const int s0 = __shfl_sync(full, gp0, sidx), s1 = __shfl_sync(full, gp1, sidx);
                    const int sw = (s0 != g0) + (s1 != g1);
                    const int v = dv + 32 * sw + (sw ? 8 : 0);
                    if (v < best) { best = v; arg = sidx; }
                }
                Dcur = allowed ? min(best + cost, DP_INF) : DP_INF;
                if (valid) back[(int64_t)q * 16 + lane] = (uint16_t)arg;
            }
            Dprev = valid ? Dcur : DP_INF; gp0 = g0; gp1 = g1; kp = kc; rw = rw_next;
        }
        // final minimum (lowest code) and backtrace; the rows of `back` and the records are loaded by the whole warp
        const int fin = (lane < kp * kp) ? Dprev : INT32_MAX;
        const int best = __reduce_min_sync(full, fin);
        int cur = __ffs(__ballot_sync(full, fin == best)) - 1;
        if (lane == 0) d.dp_cost[c] = (double)best;
        __syncwarp();
        for (int q = n_pos - 1; q >= 0; q--) {
            const uint32_t w = lane < 22 ? recw[(int64_t)q * 22 + lane] : 0u;
            const int brow = (q > 0 && lane < 16) ? back[(int64_t)q * 16 + lane] : 0;
            const int kc = (int)(__shfl_sync(full, w, 1) & 0xffu);
            const int dg = lane == 0 ? cur / kc : cur % kc;                          // lane h writes haplotype h
            const int g = (int)__shfl_sync(full, w, 2 + (lane < 2 ? dg : 0));
            const uint32_t cmw = __shfl_sync(full, w, 20 + (lane < 2 ? (dg >> 2) : 0));
            if (lane < 2) {
                d.path[(p0 + q) * 2 + lane] = g;
                d.hap_allele[(p0 + q) * 2 + lane] = (uint8_t)((cmw >> (8 * (dg & 3))) & 0xffu);
            }
            cur = __shfl_sync(full, brow, cur);
        }
    }
}

// ---------------------------------------------------------------- CSR cells of the final matrix
template <int BITS, int G>
__global__ void __launch_bounds__(256) k_write_cells(DB d) {
    const unsigned gm = grp_mask<G>();
    const int lane = lane_id(), gl = lane % G;
    const int64_t gpb = blockDim.x / G, g0 = blockIdx.x * gpb + threadIdx.x / G;
    for (int64_t f = g0; f < d.NF; f += (int64_t)gridDim.x * gpb) {
        const int c = d.fr_chain[f];
        const int i = (int)(f - d.frow_off[c]);
        const uint32_t* row = d.codes + d.code_off[c] + (int64_t)i * d.ch_words[c];
        const int first = d.fr_first[f], last = d.fr_last[f];
        int64_t base = d.cell_off[f] - d.cell_base;
        for (int bb = first; bb <= last; bb += G) {
            const int b = bb + gl;
            const uint32_t code = b <= last ? get_code(row, b, BITS) : 0u;
            const unsigned m = __ballot_sync(gm, code != 0);                 // bits of this group's lanes only
            if (code) { const int64_t o = base + __popc(m & ((1u << lane) - 1u)); d.cell_pos[o] = b; d.cell_allele[o] = (uint8_t)(code - 1); }
            base += __popc(m);
        }
    }
}

// ---------------------------------------------------------------- exclusive scan (int32 -> int64), three launches
constexpr int SCAN_BLOCK = 1024;
__global__ void __launch_bounds__(SCAN_BLOCK) k_scan_local(const int32_t* __restrict__ in, int64_t n, int64_t* __restrict__ out, int64_t* __restrict__ block_sum) {
    __shared__ int64_t s[SCAN_BLOCK];
    const int64_t x = blockIdx.x * (int64_t)SCAN_BLOCK + threadIdx.x;
    const int64_t v = x < n ? in[x] : 0;
    s[threadIdx.x] = v;
    __syncthreads();
    for (int o = 1; o < SCAN_BLOCK; o <<= 1) {
        int64_t t = threadIdx.x >= o ? s[threadIdx.x - o] : 0;
        __syncthreads();
        s[threadIdx.x] += t;
        __syncthreads();
    }
    if (x < n) out[x] = s[threadIdx.x] - v;
    if (threadIdx.x == SCAN_BLOCK - 1) block_sum[blockIdx.x] = s[threadIdx.x];
}
// exclusive scan of the block sums in place, one block: every thread owns a contiguous run
__global__ void __launch_bounds__(SCAN_BLOCK) k_scan_blocks(int64_t* block_sum, int64_t nb, int64_t* total) {
    __shared__ int64_t s[SCAN_BLOCK];
    const int64_t per = (nb + SCAN_BLOCK - 1) / SCAN_BLOCK, lo = threadIdx.x * per, hi = lo + per < nb ? lo + per : nb;
    int64_t acc = 0;
    for (int64_t x = lo; x < hi; x++) acc += block_sum[x];
    s[threadIdx.x] = acc;
    __syncthreads();
    for (int o = 1; o < SCAN_BLOCK; o <<= 1) {
        const int64_t t = threadIdx.x >= o ? s[threadIdx.x - o] : 0;
        __syncthreads();
        s[threadIdx.x] += t;
        __syncthreads();
    }
    int64_t run = s[threadIdx.x] - acc;
    for (int64_t x = lo; x < hi; x++) { const int64_t v = block_sum[x]; block_sum[x] = run; run += v; }
    if (threadIdx.x == SCAN_BLOCK - 1) *total = s[threadIdx.x];
}
__global__ void __launch_bounds__(SCAN_BLOCK) k_scan_add(int64_t* out, int64_t n, const int64_t* __restrict__ block_sum, const int64_t* __restrict__ total, int64_t base) {
    const int64_t x = blockIdx.x * (int64_t)SCAN_BLOCK + threadIdx.x;
    if (x < n) out[x] += block_sum[blockIdx.x] + base;
    if (x == 0) out[n] = *total + base;
}

// offsets of a chunk of chains, uploaded as a raw slice of the caller's array: make them start at 0
__global__ void k_rebase(int64_t* p, int64_t n, int64_t base) {
    for (int64_t x = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; x < n; x += (int64_t)gridDim.x * blockDim.x) p[x] -= base;
}

}  // namespace ahs
