// k_front.cuh — the front end (projection, stage A, boundary set, stage B, filter, read order) of ONE CHAIN PER BLOCK, out of
// shared memory.
//
// For batches whose chains fit (every chain of BASELINE configs 2-4) it replaces the kernel sequence of k_project.cuh and
// calls the same rule functions.  What differs is where the data lives and how the work is dealt out:
//   * ids are chain-local (an allele finds its bubble by binary search: no owner maps);
//   * the chain's slice of the alignment nodes (3/4 of the batch's bytes) arrives by ONE bulk asynchronous copy
//     (cp.async.bulk + mbarrier) while the block builds the chain's trigger table;
//   * the mask and every per-read and per-bubble array live in shared memory, and the matrix crosses HBM once, as final
//     codes (the sequence moves ~9x the matrix: memset, atomics, two scans, a rewrite);
//   * chain-level values are scal[] words and block barriers instead of d.ch_* arrays and kernel boundaries;
//   * thread 0 sorts the read order while the other warps write the results out.
#pragma once
#include "common.cuh"
#include "device_batch.cuh"
#include "k_project.cuh"

namespace ahs {

constexpr int FR_THREADS = 256;
constexpr int FR_G = 16;                              // lanes per entry / per read
constexpr size_t FR_SMEM_CAP = 96 * 1024;             // per block: at least two blocks per SM

struct FrLayout { uint32_t enode, eoff, aoff, tab, arec, inc, rankA, univ, poscov, mask, ckey, ckeyA, fent, good, rdA, rd, pass, ord, okey, scal, total; };

// byte offsets of a chain's arrays inside the block's dynamic shared memory (identical on host and device)
__host__ __device__ inline FrLayout fr_layout(int B, int R, int NA, int NE, int NEN, int hcap) {
    FrLayout o; uint32_t p = 0;
    auto take = [&](uint32_t bytes, uint32_t align) { p = (p + align - 1) & ~(align - 1); const uint32_t at = p; p += bytes; return at; };
    o.enode = take((uint32_t)(NEN + 8) * 4, 16);       // + alignment slack of the bulk copy
    o.tab = take((uint32_t)hcap * 8, 8); o.ckey = take((uint32_t)R * 8, 8); o.ckeyA = take((uint32_t)R * 8, 8);
    o.arec = take((uint32_t)NA * 16, 16);
    o.eoff = take((uint32_t)(NE + 1) * 4, 4); o.aoff = take((uint32_t)(B + 1) * 4, 4); o.inc = take((uint32_t)NA * 4, 4);
    o.rankA = take((uint32_t)B * 4, 4); o.univ = take((uint32_t)B * 4, 4);
    o.rdA = take((uint32_t)R * 16, 16); o.rd = take((uint32_t)R * 16, 16); o.fent = take((uint32_t)R * 4, 4);
    o.ord = take((uint32_t)R * 4, 4); o.okey = take((uint32_t)R * 4, 4); o.scal = take(64, 8);
    o.mask = take((uint32_t)((size_t)R * B * 2 + 4), 4);
    o.good = take((uint32_t)R, 1); o.pass = take((uint32_t)R, 1); o.poscov = take((uint32_t)B, 1);
    o.total = (p + 15) & ~15u;
    return o;
}

__device__ __forceinline__ uint32_t fr_smem_addr(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// scal[]: 0 maxpos 1 flags 2 T 3 nfinal 4 status 5 npos 6,7 cells (u64) 8 work item 9 err
// chains [c_begin, c_end): one launch per range of chains with a similar shared-memory need (the chains arrive largest first)
__global__ void __launch_bounds__(FR_THREADS, 5) k_chain_front(DB d, int c_begin, int c_end, int32_t* __restrict__ work_counter) {
    extern __shared__ __align__(16) unsigned char fr_sm[];
    __shared__ __align__(8) unsigned long long s_bar;
    __shared__ int s_item;
    __shared__ FrLayout s_layout;
    const int tid = threadIdx.x, lane = tid & 31;
    const unsigned gm = grp_mask<FR_G>();
    const int gl = lane % FR_G, grp = tid / FR_G;
    constexpr int NG = FR_THREADS / FR_G;
    uint32_t bar_phase = 0;
    if (tid == 0) { asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(fr_smem_addr(&s_bar))); asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
    __syncthreads();
    long long cells_block = 0;
    while (true) {
        __syncthreads();
        if (tid == 0) s_item = atomicAdd(work_counter, 1);
        __syncthreads();
        const int c = c_begin + s_item;
        if (c >= c_end) break;
        if (*(volatile const int32_t*)d.err_flags) break;             // a malformed batch: nothing is touched (k_validate ran first)
        const int64_t b0g = d.bubble_off[c];
        const int B = (int)(d.bubble_off[c + 1] - b0g);
        const int64_t r0g = d.read_off[c];
        const int R = (int)(d.read_off[c + 1] - r0g);
        if (B <= 1) {                                                  // trivial chain: never phased (:86)
            for (int r = tid; r < R; r += FR_THREADS) d.rd_pass[r0g + r] = 0;
            if (tid == 0) { d.ch_status[c] = AHS_CHAIN_TRIVIAL; d.ch_T[c] = 0; d.ch_nfinal[c] = 0; d.ch_npos[c] = 0; d.ch_cells[c] = 0; }
            for (int b = tid; b < B; b += FR_THREADS) d.poscov[b0g + b] = 0;
            continue;
        }
        const int64_t a0 = d.allele_off[b0g];
        const int NA = (int)(d.allele_off[b0g + B] - a0);
        const int64_t e0 = d.entry_off[c];
        const int NE = (int)(d.entry_off[c + 1] - e0);
        const int64_t en0 = d.enode_off[e0];
        const int NEN = (int)(d.enode_off[e0 + NE] - en0);
        const uint32_t hmask = d.hmaskc[c];
        if (tid == 0) s_layout = fr_layout(B, R, NA, NE, NEN, (int)hmask + 1);       // once per chain, not per thread
        __syncthreads();
        const FrLayout& L = s_layout;
        int32_t* enode_s = (int32_t*)(fr_sm + L.enode); int32_t* eoff = (int32_t*)(fr_sm + L.eoff); int32_t* aoff = (int32_t*)(fr_sm + L.aoff);
        unsigned long long* tab = (unsigned long long*)(fr_sm + L.tab); int4* arec = (int4*)(fr_sm + L.arec); int32_t* inc = (int32_t*)(fr_sm + L.inc);
        int32_t* rankA = (int32_t*)(fr_sm + L.rankA); uint32_t* univ = (uint32_t*)(fr_sm + L.univ); uint8_t* poscov = fr_sm + L.poscov;
        uint16_t* mask = (uint16_t*)(fr_sm + L.mask);
        unsigned long long* ckey = (unsigned long long*)(fr_sm + L.ckey); unsigned long long* ckeyA = (unsigned long long*)(fr_sm + L.ckeyA);
        uint32_t* fent = (uint32_t*)(fr_sm + L.fent); uint8_t* good_r = fr_sm + L.good;
        int4* rdA = (int4*)(fr_sm + L.rdA);                              // {cnt, first, last, mapq}
        int4* rd = (int4*)(fr_sm + L.rd);                                // {nv, first, last, mapq}
        uint8_t* pass = fr_sm + L.pass; int32_t* ord = (int32_t*)(fr_sm + L.ord); int32_t* okey = (int32_t*)(fr_sm + L.okey);
        int32_t* scal = (int32_t*)(fr_sm + L.scal);
        const float* ident = d.entry_identity + e0;
        // ---- S0: the chain's alignment nodes by one bulk copy; everything else initialised meanwhile
        const int lead = (int)(en0 & 3);                                // the copy starts at the 16-byte boundary below the slice
        if (tid == 0 && NEN > 0) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");      // the previous chain's generic accesses to this memory come first
            const uint32_t bytes = (uint32_t)((lead + NEN) * 4 + 15) & ~15u;
            asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(fr_smem_addr(&s_bar)), "r"(bytes) : "memory");
            asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                         ::"r"(fr_smem_addr(enode_s)), "l"(d.enode + (en0 - lead)), "r"(bytes), "r"(fr_smem_addr(&s_bar)) : "memory");
        }
        for (int i = tid; i <= NE; i += FR_THREADS) eoff[i] = (int)(d.enode_off[e0 + i] - en0) + lead;
        for (int i = tid; i <= B; i += FR_THREADS) aoff[i] = (int)(d.allele_off[b0g + i] - a0);
        for (int i = tid; i <= (int)hmask; i += FR_THREADS) tab[i] = SLOT_EMPTY;
        for (int b = tid; b < B; b += FR_THREADS) { univ[b] = 0xffffffffu; rankA[b] = -1; poscov[b] = 0; }
        for (int i = tid; i < (R * B + 1) / 2 + 1; i += FR_THREADS) ((uint32_t*)mask)[i] = 0;
        for (int r = tid; r < R; r += FR_THREADS) { ckey[r] = KEY_NONE; ckeyA[r] = KEY_NONE; fent[r] = 0xffffffffu; good_r[r] = 0; pass[r] = 0; }
        if (tid < 16) scal[tid] = tid == 0 ? -1 : 0;
        __syncthreads();
        // stage-A visit ranks and the input checks of the sequence's k_validate_owned / k_rank_a / k_validate_perm
        {
            const int32_t* order = d.stage_a_order ? d.stage_a_order + b0g : nullptr;
            for (int ob = tid; ob < B; ob += FR_THREADS) if (!rank_a_store(rankA, order, ob, B)) scal[9] = 16;
        }
        for (int e = tid; e < NE; e += FR_THREADS) if (!entry_read_ok(d.entry_read[e0 + e], R)) scal[9] = 8;
        __syncthreads();
        for (int b = tid; b < B; b += FR_THREADS) if (rankA[b] < 0) scal[9] = 16;
        __syncthreads();
        if (scal[9]) { if (tid == 0) atomicOr(d.err_flags, scal[9]); if (NEN > 0) { while (true) { uint32_t ok; asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(fr_smem_addr(&s_bar)), "r"(bar_phase) : "memory"); if (ok) break; } bar_phase ^= 1; } continue; }
        // ---- S1: trigger table of the chain
        for (int ga = tid; ga < NA; ga += FR_THREADS) {
            int lo = 0, hi = B - 1;                                     // bubble of the allele
            while (lo < hi) { const int mid = (lo + hi) >> 1; if (aoff[mid + 1] > ga) hi = mid; else lo = mid + 1; }
            const int64_t o = d.anode_off[a0 + ga];
            allele_insert(arec, inc, tab, hmask, &univ[lo], &scal[1], ga, lo, ga - aoff[lo], d.anode + o, (int)(d.anode_off[a0 + ga + 1] - o), rankA[lo]);
        }
        __syncthreads();
        if (NEN > 0) {                                                  // the alignment nodes have landed
            while (true) { uint32_t ok; asm volatile("{ .reg .pred p; mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2; selp.u32 %0, 1, 0, p; }" : "=r"(ok) : "r"(fr_smem_addr(&s_bar)), "r"(bar_phase) : "memory"); if (ok) break; }
            bar_phase ^= 1;
        }
        // ---- S2: projection, one group of FR_G lanes per entry
        for (int e = grp; e < NE; e += NG) {
            const int rl = d.entry_read[e0 + e];
            const bool good = good_identity(ident[e]);
            uint64_t ck, ckA;
            project_entry<FR_G, false>(enode_s + eoff[e], eoff[e + 1] - eoff[e], tab, hmask, arec, inc, d.anode_off + a0, d.anode, mask + rl * B,
                                       good, (uint32_t)e, gm, ck, ckA);
            if (gl == 0) {
                atomicMin(&fent[rl], (uint32_t)e); if (good) good_r[rl] = 1;
                if (ck != KEY_NONE) atomicMin(&ckey[rl], (unsigned long long)ck);
                if (ckA != KEY_NONE) atomicMin(&ckeyA[rl], (unsigned long long)ckA);
            }
        }
        __syncthreads();
        // ---- S3: stage-A statistics per read
        for (int r = grp; r < R; r += NG) {
            const int3 s = stage_a_row<FR_G>(mask + r * B, B, gl, gm);
            if (gl == 0) {
                int mapq = 0;
                if (s.x > 0) { mapq = key_mapq(ident, ckeyA[r]); atomicMax(&scal[0], s.z); }
                rdA[r] = make_int4(s.x, s.y, s.z, mapq);
            }
        }
        __syncthreads();
        // ---- S4: boundary flags, to_be_added = [0, T)
        for (int r = tid; r < R; r += FR_THREADS) {
            const int4 q = rdA[r];
            if (!read_passes(q.x, q.w)) continue;
            const int f = boundary_flags(q.y, q.z, scal[0]);
            if (f) atomicOr(&scal[1], f);
        }
        __syncthreads();
        if (tid == 0) scal[2] = chain_T(scal[0], scal[1], B, scal[4]);
        __syncthreads();
        // ---- S5: final rows per read
        {
            const int T = scal[2];
            const bool live = scal[4] == AHS_CHAIN_OK;
            const uint32_t* univ_c = (scal[1] & CH_HAS_UNIV) ? univ : nullptr;
            for (int r = grp; r < R; r += NG) {
                if (!live) { if (gl == 0) { rd[r] = make_int4(0, INT32_MAX, -1, 0); pass[r] = 0; } continue; }
                uint64_t ck = ckey[r];
                const RowOut o = final_row<FR_G>(mask + r * B, B, T, univ_c, fent[r], good_r[r] != 0, ck, ident, poscov, gl, gm);
                if (gl == 0) {
                    rd[r] = make_int4(o.nv, o.first, o.last, o.mapq); pass[r] = o.pass ? 1 : 0; ckey[r] = ck;
                    if (o.pass) { atomicAdd(&scal[3], 1); atomicAdd((unsigned long long*)&scal[6], (unsigned long long)o.nv); }
                }
            }
        }
        __syncthreads();
        // ---- S6: read order, then ReadSet::sort() replayed; positions
        for (int r = tid; r < R; r += FR_THREADS) {
            if (!pass[r]) continue;
            const int rank = creation_rank(pass, (const uint64_t*)ckey, R, ckey[r]);
            ord[rank] = r; okey[rank] = rd[r].y;
        }
        __syncthreads();
        // thread 0 replays the sort (serial by nature) while the other warps write the matrix and the per-read results out
        if (tid == 0 && scal[4] == AHS_CHAIN_OK) {
            const int n = scal[3];
            if (n == 0) scal[4] = AHS_CHAIN_EMPTY;                                     // :279-282
            else if (n > 16) { KV a; a.k = okey; a.v = ord; kv_std_sort<false>(a, n); }      // up to 16 keys: insertion sort of an ascending sequence, the identity (A#22)
        }
        if (tid >= 32 && tid < 64) {
            int np = 0;
            for (int b = lane; b < B; b += 32) np += poscov[b] ? 1 : 0;
            np = warp_sum_i32(np);
            if (lane == 0) scal[5] = np;
        }
        // ---- S7: results to HBM: the matrix once, as final codes
        if (tid >= 32) {
            uint32_t* gmask = (uint32_t*)(d.mask + d.mrow_off[c]);                    // chain bases are 4-byte aligned
            const int words = (R * B + 1) / 2;
            for (int i = tid - 32; i < words; i += FR_THREADS - 32) gmask[i] = ((uint32_t*)mask)[i];
            for (int r = tid - 32; r < R; r += FR_THREADS - 32) {
                const int4 q = rd[r];
                d.rd_nv[r0g + r] = q.x; d.rd_first[r0g + r] = q.y; d.rd_last[r0g + r] = q.z; d.rd_mapq[r0g + r] = q.w; d.rd_pass[r0g + r] = pass[r];
            }
            for (int b = tid - 32; b < B; b += FR_THREADS - 32) d.poscov[b0g + b] = poscov[b];
        }
        __syncthreads();
        {
            const int n = scal[3];
            for (int i = tid; i < n; i += FR_THREADS) { d.ord[r0g + i] = ord[i]; d.okey[r0g + i] = okey[i]; }
            if (tid == 0) {
                d.ch_status[c] = scal[4]; d.ch_maxpos[c] = scal[0]; d.ch_flags[c] = scal[1]; d.ch_T[c] = scal[2];
                d.ch_nfinal[c] = n; d.ch_npos[c] = scal[5];
                const unsigned long long cells = *(unsigned long long*)&scal[6];
                d.ch_cells[c] = cells; cells_block += (long long)cells;
            }
        }
    }
    if (tid == 0 && cells_block) atomicAdd((unsigned long long*)d.tot_cells, (unsigned long long)cells_block);
}

}  // namespace ahs
