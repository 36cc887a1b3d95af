/*
 * ahsoka_b200.h — C ABI of the B200-native phasing hot path.
 *
 * This is the drop-in boundary for the single call
 *     alignmentsToReadset(alignmentreader, graph, chainpathToAlleles, readsetfile,
 *                         logging, size_sorting, g_display_mutex)
 * at reference src/polyassembly.cpp:171 (signature: src/alignmentstoreadset.cpp:55).
 * The caller keeps GFA/GAF parsing, bubble/chain detection and allele-path
 * enumeration (reference src/graph.cpp, src/alignmentreader.cpp,
 * src/chainstoreadset.cpp), flattens their containers into the CSR-by-chain batch
 * below, calls ahs_phase_batch(), and writes the result text exactly as
 * src/alignmentstoreadset.cpp:70-83 and :411-486 do.  See INTEGRATION.md.
 *
 * Plain C: pointers and sizes only, no exceptions cross the boundary.  State kept between
 * calls, per device: the CUDA context, streams and memory pools (reused by the next call) and
 * the result buffers of the LAST call, which the caller owns until ahs_free_out().
 *
 * One outstanding result per device: ahs_phase_batch() on a device whose previous
 * ahs_batch_out has not been released returns AHS_ERR_ARG (the result arrays live in a
 * per-device page-locked pool).  Calls on different devices may run concurrently from
 * different host threads; calls on one device are serialised by the library.
 */
#ifndef AHSOKA_B200_H
#define AHSOKA_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define AHS_ABI_VERSION 3   /* 3: ahs_phase_batch_genotyped */

/* Return codes of the entry points. */
#define AHS_OK              0
#define AHS_ERR_ARG         1   /* malformed batch (offsets not monotone, ploidy unsupported, ...) */
#define AHS_ERR_CUDA        2   /* CUDA runtime error or no usable device: the GPU path is mandatory */
#define AHS_ERR_LIMIT       3   /* a size limit of this build was exceeded (see ahs_limits) */
#define AHS_ERR_INTERNAL    4

/* Per-chain status (ahs_batch_out.status). */
#define AHS_CHAIN_OK            0   /* phased: path / hap_allele are valid */
#define AHS_CHAIN_TRIVIAL       1   /* <= 1 bubble: header only (alignmentstoreadset.cpp:86) */
#define AHS_CHAIN_EMPTY         2   /* no read survives the filter (alignmentstoreadset.cpp:279-282) */
#define AHS_CHAIN_TOO_LARGE     3   /* exceeds a build limit (cluster editing workspace, DP states) */
#define AHS_CHAIN_SORT_FALLBACK 4   /* ABI 1 only: never produced since ABI 2 (std::sort's heap-sort fall-back is replayed too) */

/*
 * Input batch, caller-owned, read-only, host memory.  CSR by chain.
 *
 * Chains appear in the order the reference processes them (size_sorting,
 * polyassembly.cpp:136-140).  Bubble b of chain c (b = the reference's bubble id =
 * the DP "position") is global bubble  bubble_off[c] + b.
 *
 * Alignment entries are the elements of alignmentreader.alignments[chain]
 * (alignmentreader.hpp:38) in vector order; consecutive identical entries (the
 * per-node duplication of alignmentreader.cpp:176-183) may be dropped by the
 * caller, the result is the same (alignmentstoreadset.cpp:127,245).
 */
typedef struct ahs_batch_in {
    int32_t        n_chains;
    int32_t        ploidy;          /* reference: 2 (alignmentstoreadset.cpp:306) */
    const int32_t *chain_id;        /* [n_chains] reference chain ids (opaque, echoed) */

    const int64_t *bubble_off;      /* [n_chains+1] -> global bubble index */
    const int64_t *allele_off;      /* [n_bubbles+1] -> global allele index; allele index within the
                                       bubble = position in pathToAlleles[chain][bubble] */
    const int64_t *anode_off;       /* [n_alleles+1] -> anode */
    const int32_t *anode;           /* allele-path node ids, path order kept (first and last are
                                       dropped for the inner-containment test, :510-511) */
    const int32_t *stage_a_order;   /* [n_bubbles] per chain a permutation of its bubble ids: the order
                                       in which stage A visits bubbles (unordered_map iteration,
                                       :90).  NULL = descending bubble id. */

    const int64_t *read_off;        /* [n_chains+1] -> number of distinct read names per chain */
    const int64_t *entry_off;       /* [n_chains+1] -> global entry index */
    const int64_t *enode_off;       /* [n_entries+1] -> enode */
    const int32_t *enode;           /* raw node ids of the alignment path (unsorted, may repeat) */
    const int32_t *entry_read;      /* [n_entries] chain-local read index, numbered in order of first
                                       appearance within the chain's entry list */
    const float   *entry_identity;  /* [n_entries] AlignmentPath::id as parsed by stof */
} ahs_batch_in;

/*
 * Output batch, library-allocated (host memory), released with ahs_free_out().
 * "final reads" = rows of the read x bubble allele matrix after stage B, the
 * (>=2 variants, mapq>=93) filter and ReadSet::sort()  (:210-297).
 */
typedef struct ahs_batch_out {
    int32_t   n_chains;
    int32_t   ploidy;
    int32_t  *status;        /* [n_chains] AHS_CHAIN_* */

    int64_t  *read_off;      /* [n_chains+1] -> final reads */
    int32_t  *read_id;       /* [n_reads] chain-local read index (ahs_batch_in.entry_read numbering) */
    int32_t  *read_mapq;     /* [n_reads] int(float(id)*100) of the entry that created the read */
    int32_t  *read_cluster;  /* [n_reads] cluster id within the chain (ClusterEditingSolution) */
    int64_t  *cell_off;      /* [n_reads+1] -> cells of each read, ascending position */
    int32_t  *cell_pos;      /* [n_cells] bubble id */
    uint8_t  *cell_allele;   /* [n_cells] allele index */

    int32_t  *n_clusters;    /* [n_chains] */
    int64_t  *pos_off;       /* [n_chains+1] -> covered positions (ReadSet::get_positions) */
    int32_t  *pos;           /* [n_pos] bubble ids, ascending per chain */
    int32_t  *path;          /* [n_pos * ploidy] path[j][h] = global cluster id (computePaths, :408) */
    uint8_t  *hap_allele;    /* [n_pos * ploidy] new_consensus[j][path[j][h]] (:420-423) */
    double   *dp_cost;       /* [n_chains] minimum threading cost (integer valued) */

    /* Stage-A by-products kept for the -readset dumps and tests. */
    int32_t  *maxpos;        /* [n_chains] largest fully contained bubble id, -1 if none (:193) */

    /* Work counters (the units of BASELINE.json's metric). */
    int64_t   n_cells;       /* non-missing entries of the final matrices */
    int64_t   n_pairs;       /* read pairs (i<j, same chain) sharing >= 1 position */
    int64_t   n_chains_ok;   /* chains with status 0 */

    /* Device-side timings of the last call, milliseconds (CUDA events). */
    float     ms_h2d, ms_project, ms_rows, ms_score, ms_cluster, ms_consensus, ms_thread, ms_d2h;
    float     ms_total_device;   /* first kernel start -> last kernel end, inputs resident */
    int32_t   n_launches;        /* kernels launched per pass over the batch */
    int32_t   reserved;          /* library-private (how ahs_free_out releases this result); do not touch */
    /* Algorithmic byte counts of the last call (SURVEY.md §8d formulas), for roofline reports. */
    int64_t   bytes_project, bytes_score, bytes_consensus;
} ahs_batch_out;

/* Build limits, so callers can size work and tests can probe the edges. */
typedef struct ahs_limits {
    int32_t max_ploidy;            /* largest ploidy the threading kernel accepts */
    int32_t max_alleles;           /* alleles per bubble (4-bit codes: 15) */
    int32_t max_reads_cluster;     /* final reads per chain accepted by cluster editing */
    int32_t max_positions;         /* bubbles per chain */
    int32_t max_clusters_position; /* clusters present at one position (coverage / consensus stage); more ->
                                      AHS_CHAIN_TOO_LARGE for that chain */
    int32_t reserved[3];
} ahs_limits;

int  ahs_abi_version(void);
void ahs_get_limits(ahs_limits *out);

/* Number of CUDA devices visible; <= 0 means the library cannot run (no CPU path exists). */
int  ahs_device_count(void);

/*
 * Phase one batch on one device.  Blocking.  `device` is a CUDA ordinal.
 * Host buffers in, host buffers out: H2D and D2H are inside the call.
 * Returns AHS_OK or an AHS_ERR_* code; ahs_last_error() gives the text.
 */
int  ahs_phase_batch(const ahs_batch_in *in, ahs_batch_out *out, int device);

/*
 * Phase one batch across `n_devices` devices of this process (device_ids[0..n)).
 * Chains are independent (alignmentstoreadset.cpp:75): every device gets one
 * contiguous share of them, balanced by ahs_chain_cost, and runs on its own host
 * thread and streams; there is no inter-GPU traffic; every device writes its
 * results straight into its slices of the output arrays, in input order.
 */
int  ahs_phase_batch_multi(const ahs_batch_in *in, ahs_batch_out *out,
                           const int *device_ids, int n_devices);

/*
 * Phase one batch with caller-supplied genotypes.  n_devices == 1: as ahs_phase_batch on
 * device_ids[0]; more: as ahs_phase_batch_multi, with the same shares.
 *
 * allele_dosage[n_alleles] is indexed like allele_off: allele a of global bubble gb is entry
 * allele_off[gb] + a, and holds the number of haplotypes that carry that allele.  Per bubble, either
 * every dosage is 0 (genotype unknown) or the dosages sum to `ploidy`; anything else, at any bubble
 * (trivial chains and bubbles no read covers included), fails the whole call with AHS_ERR_ARG and a
 * message naming allele_dosage, and no chain is phased.
 *
 * Where the genotype of a covered position is known, the threading DP allows only the states whose
 * multiset of consensus alleles equals {a: dosage[a] : dosage[a] > 0} (the consensus the threader
 * receives: clusters in ascending id order); where it is unknown the built-in rule applies
 * ({0:1, 1:1} at ploidy 2, "the consensus alleles are not all equal" above).  If no state of a
 * column conforms, every state is allowed.  Costs and tie rules are those of ahs_phase_batch, so the
 * emitted hap_allele multiset may still differ from the genotype.  allele_dosage == NULL, or all
 * zero, gives the result of ahs_phase_batch / ahs_phase_batch_multi bit for bit.
 */
int  ahs_phase_batch_genotyped(const ahs_batch_in *in, const uint8_t *allele_dosage,
                               ahs_batch_out *out, const int *device_ids, int n_devices);

/*
 * Resident-input variant used for device-only timing: upload once, run the kernels
 * `iters` times on the resident copy, download once.  Same results as ahs_phase_batch.
 * out->ms_* hold the average per-iteration kernel times.
 */
int  ahs_phase_batch_resident(const ahs_batch_in *in, ahs_batch_out *out, int device,
                              int warmup, int iters);

void ahs_free_out(ahs_batch_out *out);

/*
 * Optional: create the device context (CUDA context, streams, kernel attributes, tables) and reserve
 * `device_bytes` of device memory (a pass uses ~5.5x the bytes of enode[]) and `pinned_bytes` of
 * page-locked result memory (~0.6x enode[]) ahead of the first
 * ahs_phase_batch on `device`, e.g. from a second host thread while the caller still parses its
 * input (the reference has no counterpart: it is what a one-shot CLI process pays once, ~0.3-3 s).
 * Thread-safe against ahs_phase_batch; zero sizes reserve nothing.
 */
int  ahs_warmup(int device, uint64_t device_bytes, uint64_t pinned_bytes);

/* Page-lock / unlock a caller buffer so that the H2D copies inside ahs_phase_batch run at full
 * PCIe speed (optional; plain cudaHostRegister / cudaHostUnregister). */
int  ahs_pin_host(const void *ptr, uint64_t bytes);
int  ahs_unpin_host(const void *ptr);

const char *ahs_last_error(void);

/*
 * Diagnostic: sort n (key, value) pairs in place exactly as libstdc++'s std::sort does with a comparator that
 * looks at the key only (ascending, or descending if `descending` != 0) — the device routine that replays
 * ReadSet::sort() (alignmentstoreadset.cpp:297) and the cluster sort (:720), heap-sort fall-back included.
 * Host arrays in, host arrays out; runs one device thread.  For the parity tests.
 */
int  ahs_debug_std_sort(int32_t *keys, int32_t *values, int32_t n, int descending, int device);

/* Cost model used to balance the devices' shares (streaming + cluster editing + DP work), exposed for the host tools. */
double ahs_chain_cost(int64_t n_bubbles, int64_t n_entries, int64_t n_entry_nodes, int ploidy);

/*
 * The share rule of ahs_phase_batch_multi, for host tools that place chains themselves (one process per GPU):
 * cuts[0..n_parts] with 0 = cuts[0] <= ... <= cuts[n_parts] = n_chains, part g = chains [cuts[g], cuts[g+1]),
 * contiguous (the chains arrive largest first, polyassembly.cpp:135-140) and such that the largest summed cost is as
 * small as contiguous cuts allow.  Host-only: needs no CUDA device.  Returns AHS_OK or AHS_ERR_ARG.
 */
int  ahs_plan_shares(const double *chain_cost, int64_t n_chains, int n_parts, int64_t *cuts);

#ifdef __cplusplus
}
#endif
#endif /* AHSOKA_B200_H */
