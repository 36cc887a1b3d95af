// k_project.cuh — projection of alignment entries onto bubbles -> read x bubble allele matrix.
//
// Replaces reference src/alignmentstoreadset.cpp:90-136 (stage A), :146-209 (filter, boundary
// set), :210-254 (stage B), :262-297 (filter, ReadSet::sort()) and is_subset (:495-548).
//
// Layout in HBM (per chain c, R_c distinct read names, B_c bubbles):
//   mask[mrow_off[c] + r*B_c + b]  u16: bit a (a<15) = some entry of read r with identity*100 > 90
//                                  contains the INNER nodes of allele a of bubble b (stage B test);
//                                  bit 15 = some entry contains a FULL allele path of b (stage A).
//   Set with atomicOr, so the result does not depend on scheduling.  The few order-dependent
//   facts of the reference (which entry creates a read -> its mapq; first matching allele) are
//   recovered from 64-bit atomicMin keys (position | allele | entry index), i.e. the minimum in
//   the reference's own loop order (position asc, allele asc, entry asc).
//
// Finding matches: every allele path has one TRIGGER node (its first inner node; path[0] if it
// has no inner node).  A path can only be contained in an entry that contains its trigger, so a
// hash table trigger node -> alleles turns the reference's bubbles x alleles x entries scan into
// one lookup per entry node.  Paths without inner nodes match EVERY entry in stage B
// (std::includes of an empty range, SURVEY A#9): they are kept per bubble as `bubble_univ`.
//
// Each rule is one __device__ function below, next to the kernel of this sequence that calls it; k_chain_front
// (k_front.cuh) calls the same functions on its shared-memory copies of the chain's arrays.
#pragma once
#include "common.cuh"
#include "device_batch.cuh"

namespace ahs {

// ---------------------------------------------------------------- generic helpers
__global__ void k_owner(const int64_t* __restrict__ off, int n_owner, int64_t n_elem, int32_t* __restrict__ out) {
    for (int64_t x = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; x < n_elem; x += (int64_t)gridDim.x * blockDim.x)
        out[x] = owner_of(off, n_owner, x);
}

// ---------------------------------------------------------------- input validation (first kernel of every pass)
// err_flags bits: 1 empty allele path, 2 more than 15 alleles, 4 offsets not monotone, 8 entry_read out of
// range, 16 stage_a_order is not a permutation, 32 the allele dosages of a bubble are neither all 0 nor sum to the
// ploidy.  Every later kernel of phase 1 returns at once if a bit is set, so a malformed batch can never drive an
// out-of-bounds access; the host reports the error after sync #1.
#define AHS_BAIL_ON_ERR(d) do { if (*(volatile const int32_t*)(d).err_flags) return; } while (0)

// Genotype of one bubble as one word: dosage of allele a in bits 4a..4a+3 (15 alleles x 4 bits; a valid dosage is at most
// the ploidy, 6).  A DP state conforms iff the sum of 1 << 4 * allele over its haplotypes' consensus alleles equals the key:
// the multiset test of rule R3.  `sum` = the bubble's dosage total; key 0 = genotype unknown.
__device__ __forceinline__ uint64_t genotype_key(const uint8_t* __restrict__ dosage, int k, int& sum) {
    uint64_t key = 0; sum = 0;
    for (int a = 0; a < k; a++) { const uint32_t v = dosage[a]; sum += (int)v; key += (uint64_t)(v & 15u) << (4 * a); }
    return key;
}

__global__ void k_validate(DB d, int32_t* __restrict__ max_k) {
    const int64_t stride = (int64_t)gridDim.x * blockDim.x, x0 = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
    int bad = 0, mk = 0;
    for (int64_t b = x0; b < d.NB; b += stride) {
        const int64_t k = d.allele_off[b + 1] - d.allele_off[b];
        if (k < 0) bad |= 4; else if (k > MAX_ALLELES) bad |= 2; else mk = max(mk, (int)k);
        if (d.allele_dosage && k >= 0 && k <= MAX_ALLELES && d.allele_off[b] >= 0 && d.allele_off[b + 1] <= d.NA) {
            int sum; genotype_key(d.allele_dosage + d.allele_off[b], (int)k, sum);
            if (sum != 0 && sum != d.ploidy) bad |= 32;
        }
    }
    for (int64_t a = x0; a < d.NA; a += stride) { const int64_t l = d.anode_off[a + 1] - d.anode_off[a]; if (l < 0) bad |= 4; else if (l == 0) bad |= 1; }
    for (int64_t e = x0; e < d.NE; e += stride) if (d.enode_off[e + 1] < d.enode_off[e]) bad |= 4;
    mk = warp_max_i32(mk);
    if (lane_id() == 0 && mk) atomicMax(max_k, mk);
    if (bad) atomicOr(d.err_flags, bad);
}

// an entry's read index names one of the R reads of its chain (err bit 8 otherwise)
__device__ __forceinline__ bool entry_read_ok(int32_t r, int64_t R) { return r >= 0 && r < R; }

// needs entry_chain
__global__ void k_validate_owned(DB d) {
    int bad = 0;
    for (int64_t e = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; e < d.NE; e += (int64_t)gridDim.x * blockDim.x) {
        const int c = d.entry_chain[e];
        if (!entry_read_ok(d.entry_read[e], d.read_off[c + 1] - d.read_off[c])) bad = 8;
    }
    if (bad) atomicOr(d.err_flags, bad);
}

// stage-A visit rank of bubble ob of a chain of B bubbles (inverse of stage_a_order, alignmentstoreadset.cpp:90; no order:
// last bubble first).  false: the order's value is out of range (err bit 16).  Every slot of rankA written afterwards <=>
// the order is a permutation of the chain's bubble ids.
__device__ __forceinline__ bool rank_a_store(int32_t* rankA, const int32_t* order, int ob, int B) {
    if (!order) { rankA[ob] = B - 1 - ob; return true; }
    const int32_t v = order[ob];
    if (v < 0 || v >= B) return false;
    rankA[v] = ob;
    return true;
}

__global__ void k_rank_a(DB d) {
    AHS_BAIL_ON_ERR(d);
    for (int64_t gb = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; gb < d.NB; gb += (int64_t)gridDim.x * blockDim.x) {
        const int c = d.bubble_chain[gb];
        const int64_t b0 = d.bubble_off[c];
        if (!rank_a_store(d.rankA + b0, d.stage_a_order ? d.stage_a_order + b0 : nullptr, (int)(gb - b0), (int)(d.bubble_off[c + 1] - b0)))
            atomicOr(d.err_flags, 16);
    }
}

__global__ void k_validate_perm(DB d) {
    for (int64_t gb = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; gb < d.NB; gb += (int64_t)gridDim.x * blockDim.x)
        if (d.rankA[gb] < 0) atomicOr(d.err_flags, 16);
}

// ---------------------------------------------------------------- K0: trigger table
// One open-addressing table PER CHAIN (region hoff[c], size hmaskc[c] + 1 = power of two >= 2 x alleles of the
// chain), so that all probes of a chain's entries fall into a few KB that stay in L1/L2.  Slot = (head << 32 | node
// id); all ones = empty; head = first allele of the list of alleles triggered by the node (inc_next links).
constexpr unsigned long long SLOT_EMPTY = ~0ull;

// allele a of bubble b (chain-local; ga its index into arec / inc): its 16-byte record for the projection (b | a << 20 |
// 3-node flag << 31, end nodes, stage-A rank of b), its universal-allele minimum (*univ_b and the chain flag, A#9) and
// its link into the list of its trigger node
__device__ __forceinline__ void allele_insert(int4* arec, int32_t* inc, unsigned long long* tab, uint32_t hmask, uint32_t* univ_b,
                                              int32_t* ch_flags, int32_t ga, int b, int a, const int32_t* path, int len, int32_t rank) {
    arec[ga] = make_int4((int)((uint32_t)b | ((uint32_t)a << 20) | (len == 3 ? 0x80000000u : 0u)),
                         len == 3 ? path[0] : 0, len == 3 ? path[2] : 0, rank);
    if (len <= 2) { atomicMin(univ_b, (uint32_t)a); atomicOr(ch_flags, CH_HAS_UNIV); }
    const uint32_t trig = (uint32_t)(len >= 3 ? path[1] : path[0]);
    uint32_t slot = hash_slot(trig, hmask);
    while (true) {
        const unsigned long long claimed = (0xfffffffeull << 32) | trig;          // head = -2: no allele linked yet
        const unsigned long long prev = atomicCAS(&tab[slot], SLOT_EMPTY, claimed);
        if (prev == SLOT_EMPTY || (uint32_t)prev == trig) break;
        slot = (slot + 1) & hmask;
    }
    const int32_t prev_head = atomicExch((int32_t*)&tab[slot] + 1, ga);            // little endian: high word = head
    inc[ga] = prev_head == -2 ? -1 : prev_head;
}

__global__ void k_build_triggers(DB d) {
    AHS_BAIL_ON_ERR(d);
    for (int64_t ga = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; ga < d.NA; ga += (int64_t)gridDim.x * blockDim.x) {
        const int64_t gb = d.allele_bubble[ga];
        const int c = d.bubble_chain[gb];
        const int64_t o = d.anode_off[ga];
        const int len = (int)(d.anode_off[ga + 1] - o);
        d.inc_next[ga] = -1;
        if (len <= 0) { atomicOr(d.err_flags, 1); continue; }
        if (d.bubble_off[c + 1] - d.bubble_off[c] <= 1) continue;          // trivial chain: never phased (:86)
        const int a = (int)(ga - d.allele_off[gb]);
        if (a >= MAX_ALLELES) { atomicOr(d.err_flags, 2); continue; }
        allele_insert(d.arec, d.inc_next, d.hslots + d.hoff[c], d.hmaskc[c], &d.bubble_univ[gb], &d.ch_flags[c], (int32_t)ga,
                      (int)(gb - d.bubble_off[c]), a, d.anode + o, len, d.rankA[gb]);
    }
}

// ---------------------------------------------------------------- sub-warp groups
// The per-read kernels below are latency bound (a chain of dependent metadata loads per read, then a row of ~40
// cells): G lanes per read and 32/G reads in flight per warp multiply the memory-level parallelism.  Every
// collective uses the group's own lane mask, so groups of one warp proceed independently.
template <int G> __device__ __forceinline__ unsigned grp_mask() { return G == 32 ? 0xffffffffu : (((1u << G) - 1u) << ((threadIdx.x & 31) / G * G)); }
template <int G> __device__ __forceinline__ uint64_t grp_min_u64(uint64_t v, unsigned m) {
#pragma unroll
    for (int o = G >> 1; o > 0; o >>= 1) { const uint64_t t = __shfl_xor_sync(m, v, o); v = t < v ? t : v; }
    return v;
}

// ---------------------------------------------------------------- K1: project entries
// first allele triggered by node v (head of its list), -1 if none
__device__ __forceinline__ int32_t trigger_lookup(const unsigned long long* tab, uint32_t hmask, int32_t v) {
    uint32_t slot = hash_slot((uint32_t)v, hmask);
    while (true) {
        const unsigned long long sl = tab[slot];
        if (sl == SLOT_EMPTY) return -1;
        if ((uint32_t)sl == (uint32_t)v) return (int32_t)(sl >> 32);
        slot = (slot + 1) & hmask;
    }
}

// an entry's nodes in global memory (GMEM: through the read-only cache) or in shared memory, where __ldg must not go
template <bool GMEM> __device__ __forceinline__ int32_t entry_node(const int32_t* p) {
    if constexpr (GMEM) return __ldg(p); else return *p;
}

// is value q among the L nodes of the entry?  (whole lane group)
template <int G, bool GMEM>
__device__ __forceinline__ bool entry_has(const int32_t* __restrict__ nodes, int L, int32_t q, int gl, unsigned gm) {
    bool f = false;
    for (int x = gl; x < L; x += G) f |= entry_node<GMEM>(nodes + x) == q;
    return __any_sync(gm, f);
}

// One group of G lanes projects one alignment entry (index el within its chain) onto its read's mask row; lanes stride over
// the entry's nodes.  A node that is the trigger of an allele path (hash hit) decides the two containment tests of the
// reference (is_subset with and without the end nodes, :495-548).  Common case, decided by the lane alone: a 3-node path
// whose end nodes are the neighbours of the trigger in the alignment.  Everything else is decided by the whole group
// scanning the entry.  arec, inc and anode_off are indexed by the allele ids the table holds.  Returns, on every lane of
// the group, the smallest creation keys (position | allele | entry) of the stage-B (ck) and stage-A (ckA) matches.
template <int G, bool GMEM>
__device__ __forceinline__ void project_entry(const int32_t* __restrict__ nodes, int L, const unsigned long long* tab, uint32_t hmask,
                                              const int4* arec, const int32_t* inc, const int64_t* anode_off, const int32_t* anode,
                                              uint16_t* mrow, bool good, uint32_t el, unsigned gm, uint64_t& ck_out, uint64_t& ckA_out) {
    const int lane = lane_id(), gl = lane % G;
    uint64_t ck = KEY_NONE, ckA = KEY_NONE;                 // smallest creation keys seen by this lane
    for (int x0 = 0; x0 < L; x0 += G) {
        const int x = x0 + gl;
        int32_t ga = -1, prev = 0, next = 0; bool has_prev = false, has_next = false;
        if (x < L) {
            has_prev = x > 0; has_next = x + 1 < L;
            if (has_prev) prev = entry_node<GMEM>(nodes + x - 1);
            if (has_next) next = entry_node<GMEM>(nodes + x + 1);
            ga = trigger_lookup(tab, hmask, entry_node<GMEM>(nodes + x));
        }
        while (__any_sync(gm, ga >= 0)) {
            const bool have = ga >= 0;
            int64_t o = 0; int len = 0;
            bool inner_ok = false, full_ok = false, slow = false;
            int4 rec = make_int4(0, 0, 0, 0);
            if (have) {
                rec = arec[ga];
                if (rec.x < 0) {                                                      // 3-node path
                    inner_ok = true;                                                  // the only inner node is the trigger
                    full_ok = has_prev && has_next && ((prev == rec.y && next == rec.z) || (prev == rec.z && next == rec.y));
                    slow = !full_ok;                                                  // the end nodes may still be elsewhere in the entry
                } else slow = true;
                if (slow) { o = anode_off[ga]; len = (int)(anode_off[ga + 1] - o); }
            }
            for (unsigned sm = __ballot_sync(gm, slow); sm; sm &= sm - 1) {
                const int src_lane = __ffs(sm) - 1;                                   // absolute lane, inside this group
                const int64_t oo = __shfl_sync(gm, o, src_lane);
                const int ll = __shfl_sync(gm, len, src_lane);
                bool in_ok = ll >= 3;                          // len <= 2: universal, handled by final_row
                for (int y = 2; in_ok && y < ll - 1; y++) in_ok = entry_has<G, GMEM>(nodes, L, anode[oo + y], gl, gm);
                bool f_ok;
                if (ll >= 3) f_ok = in_ok && entry_has<G, GMEM>(nodes, L, anode[oo], gl, gm) && entry_has<G, GMEM>(nodes, L, anode[oo + ll - 1], gl, gm);
                else f_ok = (ll == 1) || entry_has<G, GMEM>(nodes, L, anode[oo + 1], gl, gm);
                if (lane == src_lane) { inner_ok = in_ok; full_ok = f_ok; }
            }
            if (have) {
                const int b = (int)((uint32_t)rec.x & 0xfffffu);
                const int a = (int)(((uint32_t)rec.x >> 20) & 0xffu);
                const uint32_t bits = ((inner_ok && good) ? (1u << a) : 0u) | (full_ok ? 0x8000u : 0u);
                if (bits) atomic_or_u16(&mrow[b], (uint16_t)bits);                   // one atomic for both tests
                if (inner_ok) { const uint64_t k = make_key((uint32_t)b, (uint32_t)a, el); ck = k < ck ? k : ck; }
                if (full_ok) { const uint64_t k = make_key((uint32_t)rec.w, (uint32_t)a, el); ckA = k < ckA ? k : ckA; }
                ga = inc[ga];
            }
        }
    }
    ck_out = grp_min_u64<G>(ck, gm); ckA_out = grp_min_u64<G>(ckA, gm);
}

template <int G>
__global__ void __launch_bounds__(256, 6) k_project(DB d, int64_t e_begin, int64_t e_end) {
    AHS_BAIL_ON_ERR(d);
    const unsigned gm = grp_mask<G>();
    const int gl = lane_id() % G;
    const int64_t gpb = blockDim.x / G, g0 = blockIdx.x * gpb + threadIdx.x / G;
    for (int64_t ge = e_begin + g0; ge < e_end; ge += (int64_t)gridDim.x * gpb) {
        const int c = d.entry_chain[ge];
        const int64_t b0 = d.bubble_off[c];
        const int B = (int)(d.bubble_off[c + 1] - b0);
        if (B <= 1) continue;
        const int rl = d.entry_read[ge];
        const int64_t r = d.read_off[c] + rl;
        const uint32_t el = (uint32_t)(ge - d.entry_off[c]);
        const bool good = good_identity(d.entry_identity[ge]);
        uint64_t ck, ckA;
        project_entry<G, true>(d.enode + d.enode_off[ge], (int)(d.enode_off[ge + 1] - d.enode_off[ge]), d.hslots + d.hoff[c], d.hmaskc[c],
                               d.arec, d.inc_next, d.anode_off, d.anode, d.mask + d.mrow_off[c] + (int64_t)rl * B, good, el, gm, ck, ckA);
        if (gl == 0) {
            atomicMin(&d.first_entry[r], el); if (good) d.has_good[r] = 1;
            if (ck != KEY_NONE) atomicMin((unsigned long long*)&d.create_key[r], (unsigned long long)ck);
            if (ckA != KEY_NONE) atomicMin((unsigned long long*)&d.createA_key[r], (unsigned long long)ckA);
        }
    }
}

// ---------------------------------------------------------------- K1b: stage-A statistics per read
// count / first / last fully contained bubble of a read's mask row (:146-165), reduced over the group
template <int G>
__device__ __forceinline__ int3 stage_a_row(const uint16_t* mrow, int B, int gl, unsigned gm) {
    int cnt = 0, first = INT32_MAX, last = -1;
    for (int b = gl; b < B; b += G) if (mrow[b] & 0x8000u) { cnt++; first = min(first, b); last = max(last, b); }
    return make_int3(__reduce_add_sync(gm, cnt), __reduce_min_sync(gm, first), __reduce_max_sync(gm, last));
}

// mapq of a read: that of the entry in its creation key (ident: the identities of the chain's entries; :117, :234)
__device__ __forceinline__ int32_t key_mapq(const float* ident, uint64_t key) { return mapq_of(ident[(uint32_t)(key & 0xffffffffu)]); }

// the read filter of stage A and of the final read set (:173-182, :270)
__device__ __forceinline__ bool read_passes(int n, int32_t mapq) { return n > 1 && mapq >= 93; }

template <int G>
__global__ void __launch_bounds__(256) k_read_stage_a(DB d) {
    AHS_BAIL_ON_ERR(d);
    const unsigned gm = grp_mask<G>();
    const int gl = lane_id() % G;
    const int64_t gpb = blockDim.x / G, g0 = blockIdx.x * gpb + threadIdx.x / G;
    for (int64_t r = g0; r < d.NR; r += (int64_t)gridDim.x * gpb) {
        const int c = d.read_chain[r];
        const int B = (int)(d.bubble_off[c + 1] - d.bubble_off[c]);
        if (B <= 1) continue;
        const int3 s = stage_a_row<G>(d.mask + d.mrow_off[c] + (r - d.read_off[c]) * B, B, gl, gm);
        if (gl == 0) {
            int mapq = 0;
            if (s.x > 0) { mapq = key_mapq(d.entry_identity + d.entry_off[c], d.createA_key[r]); atomicMax(&d.ch_maxpos[c], s.z); }
            d.rdA_cnt[r] = s.x; d.rdA_first[r] = s.y; d.rdA_last[r] = s.z; d.rdA_mapq[r] = mapq;
        }
    }
}

// boundary flags of a filtered stage-A read: which of maxpos-1 / maxpos are its last (1, 2) or first (4, 8) position (:173-189)
__device__ __forceinline__ int boundary_flags(int first, int last, int mp) {
    int f = 0;
    if (last == mp) f |= 1;
    if (last == mp - 1) f |= 2;
    if (first == mp) f |= 4;
    if (first == mp - 1) f |= 8;
    return f;
}

__global__ void k_chain_flags(DB d) {
    AHS_BAIL_ON_ERR(d);
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < d.NR; r += (int64_t)gridDim.x * blockDim.x) {
        const int c = d.read_chain[r];
        if (d.bubble_off[c + 1] - d.bubble_off[c] <= 1) continue;
        if (!read_passes(d.rdA_cnt[r], d.rdA_mapq[r])) continue;
        const int f = boundary_flags(d.rdA_first[r], d.rdA_last[r], d.ch_maxpos[c]);
        if (f) atomicOr(&d.ch_flags[c], f);
    }
}

// to_be_added = [0,maxpos) U {e, e+1 : e in last \ first} = [0, T) of a chain of B > 1 bubbles, from maxpos mp and the
// boundary flags f; `status` = OK, or EMPTY when no read contains a full bubble path (:173-209, SURVEY A#10)
__device__ __forceinline__ int chain_T(int mp, int f, int B, int32_t& status) {
    if (mp < 0) { status = AHS_CHAIN_EMPTY; return 0; }          // reference: UB (:193)
    const bool e_max = (f & 1) && !(f & 4);          // maxpos   in last \ first  -> adds maxpos, maxpos+1
    const bool e_m1  = (f & 2) && !(f & 8);          // maxpos-1 in last \ first  -> adds maxpos-1, maxpos
    int T = mp;
    if (e_max) T = mp + 2; else if (e_m1) T = mp + 1;
    status = AHS_CHAIN_OK;
    return min(T, B);                                  // bubble ids >= B have no alleles (:216 default-insert)
}

__global__ void k_chain_T(DB d) {
    AHS_BAIL_ON_ERR(d);
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < d.C; c += gridDim.x * blockDim.x) {
        const int B = (int)(d.bubble_off[c + 1] - d.bubble_off[c]);
        if (B <= 1) { d.ch_status[c] = AHS_CHAIN_TRIVIAL; d.ch_T[c] = 0; continue; }
        int32_t status;
        d.ch_T[c] = chain_T(d.ch_maxpos[c], d.ch_flags[c], B, status);
        d.ch_status[c] = status;
    }
}

// ---------------------------------------------------------------- K1d: final rows per read (stage B + filter)
struct RowOut { int nv, first, last, mapq; bool pass; };

// Stage B and the filter for one read, to_be_added = [0, T) (:210-254, :262-270), by the whole group.  ck: the read's
// creation key, updated with the universal alleles (univ: nullptr if the chain has none; fe: the read's first entry).
// A read created below T gets its row rewritten into allele codes and, if it passes, its positions marked in poscov;
// other rows stay as projected, because only the rows of final reads are read afterwards.
template <int G>
__device__ __forceinline__ RowOut final_row(uint16_t* mrow, int B, int T, const uint32_t* univ, uint32_t fe, bool hg, uint64_t& ck,
                                            const float* ident, uint8_t* poscov, int gl, unsigned gm) {
    if (fe != 0xffffffffu && univ) for (int b = gl; b < T; b += G) {
        const uint32_t u = univ[b];
        if (u != 0xffffffffu) { const uint64_t k = make_key((uint32_t)b, u, fe); ck = k < ck ? k : ck; }
    }
    ck = grp_min_u64<G>(ck, gm);
    RowOut o; o.nv = 0; o.first = (ck == KEY_NONE) ? INT32_MAX : (int)(ck >> 40); o.last = -1; o.mapq = 0; o.pass = false;
    uint32_t cov = 0;                                                   // this lane's covered positions b = gl + G j, j < 32
    if (o.first < T) {
        const int ac = (int)((ck >> 32) & 0xff);
        int nv = 0, last = -1;
        for (int b = gl; b < B; b += G) {
            uint32_t code = 0;
            if (b < T) {
                uint32_t m = mrow[b] & 0x7fffu;
                const uint32_t u = univ ? univ[b] : 0xffffffffu;
                if (u != 0xffffffffu && hg) m |= 1u << u;
                if (b == o.first) code = (uint32_t)ac + 1u;
                else if (m) code = (uint32_t)__ffs((int)m);             // lowest set bit = first matching allele
            }
            mrow[b] = (uint16_t)code;
            if (code) { nv++; last = max(last, b); if (b < 32 * G) cov |= 1u << (b / G); }
        }
        o.nv = __reduce_add_sync(gm, nv); o.last = __reduce_max_sync(gm, last);
        o.mapq = key_mapq(ident, ck);
        o.pass = read_passes(o.nv, o.mapq);
    }
    __syncwarp(gm);                                                     // the group's codes are written
    if (o.pass) {
        for (uint32_t m = cov; m; m &= m - 1) poscov[gl + G * (__ffs((int)m) - 1)] = 1;   // codes are only set below T
        for (int b = gl + 32 * G; b < T; b += G) if (mrow[b]) poscov[b] = 1;
    }
    return o;
}

template <int G>
__global__ void __launch_bounds__(256) k_read_rows(DB d) {
    AHS_BAIL_ON_ERR(d);
    const unsigned gm = grp_mask<G>();
    const int gl = lane_id() % G;
    const int64_t gpb = blockDim.x / G, g0 = blockIdx.x * gpb + threadIdx.x / G;
    long long cells_local = 0;
    for (int64_t r = g0; r < d.NR; r += (int64_t)gridDim.x * gpb) {
        const int c = d.read_chain[r];
        if (gl == 0) d.rd_pass[r] = 0;
        if (d.ch_status[c] != AHS_CHAIN_OK) continue;
        const int64_t b0g = d.bubble_off[c];
        const int B = (int)(d.bubble_off[c + 1] - b0g);
        const bool univ = (d.ch_flags[c] & CH_HAS_UNIV) != 0;              // rare: a bubble with an allele path of <= 2 nodes
        uint64_t ck = d.create_key[r];
        const RowOut o = final_row<G>(d.mask + d.mrow_off[c] + (r - d.read_off[c]) * B, B, d.ch_T[c], univ ? d.bubble_univ + b0g : nullptr,
                                      d.first_entry[r], d.has_good[r] != 0, ck, d.entry_identity + d.entry_off[c], d.poscov + b0g, gl, gm);
        if (gl == 0) {
            d.rd_nv[r] = o.nv; d.rd_first[r] = o.first; d.rd_last[r] = o.last; d.rd_mapq[r] = o.mapq; d.rd_pass[r] = o.pass ? 1 : 0;
            d.create_key[r] = ck;
            if (o.pass) { atomicAdd(&d.ch_nfinal[c], 1); atomicAdd(&d.ch_cells[c], (unsigned long long)o.nv); cells_local += o.nv; }
        }
    }
    // one atomic per warp on the batch-wide cell counter (a per-read atomic on one address serialises in L2)
    __syncwarp();
    for (int o = 16; o > 0; o >>= 1) cells_local += __shfl_xor_sync(0xffffffffu, cells_local, o);
    if (lane_id() == 0 && cells_local) atomicAdd((unsigned long long*)d.tot_cells, (unsigned long long)cells_local);
}

// ---------------------------------------------------------------- K1e: read order
// Insertion order of the stage-B read set = order of the creation triples: the rank of a passing read's key among the n
// reads of its chain, by counting.
__device__ __forceinline__ int creation_rank(const uint8_t* pass, const uint64_t* key, int n, uint64_t k) {
    int rank = 0;
    for (int x = 0; x < n; x++) rank += (pass[x] && key[x] < k) ? 1 : 0;
    return rank;
}

__global__ void k_read_rank(DB d) {
    AHS_BAIL_ON_ERR(d);
    for (int64_t r = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; r < d.NR; r += (int64_t)gridDim.x * blockDim.x) {
        if (!d.rd_pass[r]) continue;
        const int c = d.read_chain[r];
        const int64_t r0 = d.read_off[c];
        const int rank = creation_rank(d.rd_pass + r0, d.create_key + r0, (int)(d.read_off[c + 1] - r0), d.create_key[r]);
        d.ord[r0 + rank] = (int32_t)(r - r0);
        d.okey[r0 + rank] = d.rd_first[r];
    }
}

// libstdc++ std::sort (introsort + final insertion sort) replayed move for move on (key, value)
// pairs with a comparator that looks at the key only: ReadSet::sort() at alignmentstoreadset.cpp:297
// (comparator on firstPosition()), and the cluster sort at :720.  SURVEY A#11, A#22.
struct KV { int32_t* k; int32_t* v; };
__device__ __forceinline__ void kv_swap(KV a, int x, int y) {
    int32_t t = a.k[x]; a.k[x] = a.k[y]; a.k[y] = t; t = a.v[x]; a.v[x] = a.v[y]; a.v[y] = t;
}
template <bool DESC> __device__ __forceinline__ bool kv_less(int32_t x, int32_t y) { return DESC ? x > y : x < y; }

template <bool DESC>
__device__ void kv_unguarded_linear_insert(KV a, int last) {
    int32_t vk = a.k[last], vv = a.v[last];
    int next = last - 1;
    while (kv_less<DESC>(vk, a.k[next])) { a.k[last] = a.k[next]; a.v[last] = a.v[next]; last = next; --next; }
    a.k[last] = vk; a.v[last] = vv;
}
template <bool DESC>
__device__ void kv_insertion_sort(KV a, int first, int last) {
    if (first == last) return;
    for (int i = first + 1; i != last; ++i) {
        if (kv_less<DESC>(a.k[i], a.k[first])) {
            int32_t vk = a.k[i], vv = a.v[i];
            for (int x = i; x > first; --x) { a.k[x] = a.k[x - 1]; a.v[x] = a.v[x - 1]; }
            a.k[first] = vk; a.v[first] = vv;
        } else kv_unguarded_linear_insert<DESC>(a, i);
    }
}
// std::__adjust_heap + std::__push_heap (bits/stl_heap.h) on the sub-array starting at `first`
template <bool DESC>
__device__ void kv_adjust_heap(KV a, int first, int hole, int len, int32_t vk, int32_t vv) {
    const int top = hole;
    int child = hole;
    while (child < (len - 1) / 2) {
        child = 2 * (child + 1);
        if (kv_less<DESC>(a.k[first + child], a.k[first + child - 1])) child--;
        a.k[first + hole] = a.k[first + child]; a.v[first + hole] = a.v[first + child];
        hole = child;
    }
    if ((len & 1) == 0 && child == (len - 2) / 2) {
        child = 2 * (child + 1);
        a.k[first + hole] = a.k[first + child - 1]; a.v[first + hole] = a.v[first + child - 1];
        hole = child - 1;
    }
    int parent = (hole - 1) / 2;
    while (hole > top && kv_less<DESC>(a.k[first + parent], vk)) {
        a.k[first + hole] = a.k[first + parent]; a.v[first + hole] = a.v[first + parent];
        hole = parent; parent = (hole - 1) / 2;
    }
    a.k[first + hole] = vk; a.v[first + hole] = vv;
}
// std::__partial_sort(first, last, last): __heap_select (= __make_heap, the selection loop is empty) + __sort_heap —
// what __introsort_loop falls back to when its depth limit is used up
template <bool DESC>
__device__ void kv_heap_sort(KV a, int first, int last) {
    const int len = last - first;
    if (len < 2) return;
    for (int parent = (len - 2) / 2; ; parent--) {
        kv_adjust_heap<DESC>(a, first, parent, len, a.k[first + parent], a.v[first + parent]);
        if (parent == 0) break;
    }
    for (int end = last; end - first > 1; ) {
        --end;
        const int32_t vk = a.k[end], vv = a.v[end];
        a.k[end] = a.k[first]; a.v[end] = a.v[first];
        kv_adjust_heap<DESC>(a, first, 0, end - first, vk, vv);
    }
}
// std::sort(first, last, comp) of libstdc++ (bits/stl_algo.h: __introsort_loop with depth limit 2 lg n, then
// __final_insertion_sort), heap-sort fall-back included
template <bool DESC>
__device__ void kv_std_sort(KV a, int n) {
    if (n <= 1) return;
    int depth0 = 0; for (int m = n; m > 1; m >>= 1) depth0++;
    depth0 *= 2;
    int stk_first[64], stk_last[64], stk_depth[64]; int sp = 0;
    stk_first[0] = 0; stk_last[0] = n; stk_depth[0] = depth0; sp = 1;
    while (sp > 0) {
        --sp;
        int first = stk_first[sp], last = stk_last[sp], depth = stk_depth[sp];
        while (last - first > 16) {
            if (depth == 0) { kv_heap_sort<DESC>(a, first, last); break; }
            --depth;
            // __move_median_to_first(first, first+1, mid, last-1)
            int mid = first + (last - first) / 2, A = first + 1, Bm = mid, Cc = last - 1;
            if (kv_less<DESC>(a.k[A], a.k[Bm])) {
                if (kv_less<DESC>(a.k[Bm], a.k[Cc])) kv_swap(a, first, Bm);
                else if (kv_less<DESC>(a.k[A], a.k[Cc])) kv_swap(a, first, Cc);
                else kv_swap(a, first, A);
            } else if (kv_less<DESC>(a.k[A], a.k[Cc])) kv_swap(a, first, A);
            else if (kv_less<DESC>(a.k[Bm], a.k[Cc])) kv_swap(a, first, Cc);
            else kv_swap(a, first, Bm);
            // __unguarded_partition(first+1, last, pivot=first)
            int lo = first + 1, hi = last;
            const int32_t pk = a.k[first];
            while (true) {
                while (kv_less<DESC>(a.k[lo], pk)) ++lo;
                --hi;
                while (kv_less<DESC>(pk, a.k[hi])) --hi;
                if (!(lo < hi)) break;
                kv_swap(a, lo, hi);
                ++lo;
            }
            // recurse on [cut,last), loop on [first,cut): the right part is sorted first, but the
            // parts are disjoint, so the order of processing does not change the result.  The stack
            // cannot overflow: every push lowers `depth`, so at most depth0 <= 2 * 31 ranges are pending.
            stk_first[sp] = lo; stk_last[sp] = last; stk_depth[sp] = depth; ++sp;
            last = lo;
        }
    }
    // __final_insertion_sort
    if (n > 16) {
        kv_insertion_sort<DESC>(a, 0, 16);
        for (int i = 16; i < n; ++i) kv_unguarded_linear_insert<DESC>(a, i);
    } else kv_insertion_sort<DESC>(a, 0, n);
}

// diagnostic kernel behind ahs_debug_std_sort: one thread replays std::sort on (key, value) pairs
__global__ void k_debug_std_sort(int32_t* k, int32_t* v, int n, int desc) {
    KV a; a.k = k; a.v = v;
    if (desc) kv_std_sort<true>(a, n); else kv_std_sort<false>(a, n);
}

__global__ void k_chain_sort(DB d) {
    AHS_BAIL_ON_ERR(d);
    for (int c = blockIdx.x * blockDim.x + threadIdx.x; c < d.C; c += gridDim.x * blockDim.x) {
        if (d.ch_status[c] != AHS_CHAIN_OK) continue;
        const int n = d.ch_nfinal[c];
        if (n == 0) { d.ch_status[c] = AHS_CHAIN_EMPTY; continue; }            // :279-282
        KV a; a.k = d.okey + d.read_off[c]; a.v = d.ord + d.read_off[c];
        kv_std_sort<false>(a, n);
        // covered positions (ReadSet::get_positions, :317)
    }
}

// covered positions per chain: count, then (after the host has the offsets) the compact list
__global__ void k_count_pos(DB d) {
    AHS_BAIL_ON_ERR(d);
    const int wpb = blockDim.x >> 5, lane = lane_id();
    for (int c = blockIdx.x * wpb + (threadIdx.x >> 5); c < d.C; c += gridDim.x * wpb) {
        const int64_t b0 = d.bubble_off[c];
        const int B = (int)(d.bubble_off[c + 1] - b0);
        int n = 0;
        for (int b = lane; b < B; b += 32) n += d.poscov[b0 + b] ? 1 : 0;
        n = warp_sum_i32(n);
        if (lane == 0) d.ch_npos[c] = n;
    }
}

__global__ void k_compact_pos(DB d) {
    const int wpb = blockDim.x >> 5, lane = lane_id();
    for (int c = blockIdx.x * wpb + (threadIdx.x >> 5); c < d.C; c += gridDim.x * wpb) {
        const int64_t b0 = d.bubble_off[c];
        const int B = (int)(d.bubble_off[c + 1] - b0);
        const bool live = d.ch_status[c] == AHS_CHAIN_OK;
        int base = 0;
        for (int bb = 0; bb < B; bb += 32) {
            const int b = bb + lane;
            const bool cov = live && b < B && d.poscov[b0 + b];
            const unsigned m = __ballot_sync(0xffffffffu, cov);
            if (b < B) d.pos_compact[b0 + b] = cov ? base + __popc(m & ((1u << lane) - 1u)) : -1;
            if (cov) d.pos[d.pos_off[c] + base + __popc(m & ((1u << lane) - 1u))] = b;
            base += __popc(m);
        }
    }
}

// ---------------------------------------------------------------- K1f: pack final rows
// G lanes per final read: mask row (u16 codes) -> packed 2/4-bit codes, dense by bubble id.  Lanes read consecutive
// codes (coalesced), shift them into place and OR them together across the group, one word at a time.
template <int G>
__global__ void __launch_bounds__(256) k_pack_rows(DB d) {
    const unsigned gm = grp_mask<G>();
    const int gl = lane_id() % G;
    const int64_t gpb = blockDim.x / G, g0 = blockIdx.x * gpb + threadIdx.x / G;
    const int bits = d.bits, per_word = 32 / bits;
    for (int64_t f = g0; f < d.NF; f += (int64_t)gridDim.x * gpb) {
        const int c = d.fr_chain[f];
        const int B = (int)(d.bubble_off[c + 1] - d.bubble_off[c]);
        const int i = (int)(f - d.frow_off[c]);
        const int rl = d.ord[d.read_off[c] + i];
        const int64_t r = d.read_off[c] + rl;
        const uint16_t* mrow = d.mask + d.mrow_off[c] + (int64_t)rl * B;
        uint32_t* row = d.codes + d.code_off[c] + (int64_t)i * d.ch_words[c];
        const int first = d.rd_first[r], last = d.rd_last[r];
        for (int w = first / per_word; w <= last / per_word; w++) {
            uint32_t word = 0;
            for (int x = gl; x < per_word; x += G) { const int b = w * per_word + x; if (b < B) word |= (uint32_t)mrow[b] << (x * bits); }
            word = __reduce_or_sync(gm, word);
            if (gl == 0) row[w] = word;
        }
        if (gl == 0) {
            d.fr_first[f] = first; d.fr_last[f] = last; d.fr_mapq[f] = d.rd_mapq[r]; d.fr_id[f] = rl; d.fr_nv[f] = d.rd_nv[r];
            atomicMax(&d.ch_maxspan[c], last - first);
        }
    }
}

}  // namespace ahs
