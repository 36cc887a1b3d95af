// device_batch.cuh — the batch as it lives in HBM: one struct of device pointers handed to every
// kernel by value.  Everything is CSR-by-chain; see DESIGN.md "Data layout in HBM".
#pragma once
#include <stdint.h>
#include "../../include/ahsoka_b200.h"

namespace ahs {

// per covered position, everything the threading DP and the emission need (K3 -> K4)
struct PosRec {
    uint32_t total;          // clustered reads covering the position (coverage_sum, :686)
    uint8_t  k;              // |covMap[pos]|
    uint8_t  pad[3];
    int32_t  gid[8];         // covMap[pos][l]: global cluster ids, descending coverage (:765-775)
    uint32_t cnt_asc[8];     // count of the l-th smallest cluster id among ALL clusters at pos (:385-390, A#12)
    uint8_t  cons_asc[8];    // consensus of the l-th smallest cluster id among covMap clusters (:397-401, A#12)
    uint8_t  cons_cm[8];     // consensus of covMap[pos][l] (new_consensus[j][c_id], :422)
};

struct DB {
    int32_t C, ploidy, bits;
    int64_t NB, NA, NAN_, NR, NE, NEN, NF, NP;
    // ---- input (ahs_batch_in)
    const int64_t *bubble_off, *allele_off, *anode_off, *read_off, *entry_off, *enode_off;
    const int32_t *anode, *stage_a_order, *enode, *entry_read;
    const float   *entry_identity;
    const uint8_t *allele_dosage;       // [NA] caller genotypes (ahs_phase_batch_genotyped), null without
    // ---- owner maps
    int32_t *bubble_chain, *allele_bubble, *entry_chain, *read_chain, *rankA;
    int64_t *mrow_off;                  // [C] chain offset into mask (u16 units)
    // ---- trigger table
    unsigned long long *hslots; const int64_t *hoff; const uint32_t *hmaskc;   // per-chain hash regions (k_project.cuh)
    int32_t *inc_next; uint32_t *bubble_univ; int4 *arec;                      // arec: per-allele record read by k_project
    // ---- projection
    uint16_t *mask;
    uint64_t *create_key, *createA_key; uint32_t *first_entry; uint8_t *has_good;
    int32_t *rdA_cnt, *rdA_first, *rdA_last, *rdA_mapq;
    int32_t *rd_nv, *rd_first, *rd_last, *rd_mapq; uint8_t *rd_pass;
    int32_t *ord, *okey;
    uint8_t *poscov;
    int32_t *ch_status, *ch_maxpos, *ch_flags, *ch_T, *ch_nfinal, *ch_npos, *ch_maxspan, *ch_words, *ch_nclusters;
    int64_t *tot_cells, *tot_pairs; int32_t *err_flags;
    unsigned long long *ch_cells;                         // [C] cells of the chain's final reads
    unsigned long long *ch_pairs2;                        // [C] twice the scored pairs of a chain above CC_MAXN reads (k_read_rates): sizes its edge slots
    // ---- final reads (after the host computed the offsets)
    int64_t *frow_off, *pos_off, *code_off, *cw_off;      // [C+1],[C+1],[C],[C]
    int32_t *fr_chain, *fr_first, *fr_last, *fr_mapq, *fr_id, *fr_nv, *fr_cluster;
    uint32_t *codes;
    int32_t *pos, *pos_compact, *pos_chain;
    // ---- scoring / cluster editing
    uint16_t *es, *ed;
    const int64_t *ln, *ln1;                              // log tables, 1025 entries each
    int32_t *W;                                           // pair weights: upper triangle per chain up to CC_MAXN reads, n x n above
    uint64_t *key_scratch; int64_t *key_scratch_off;       // overflow buffers for reads with > 256 partners
    uint8_t *ch_small;                                    // [C] 1 = chain is scored + clustered out of shared memory (k_chain.cuh)
    // ---- consensus / threading
    PosRec *rec; uint16_t *back; int64_t *back_off; int32_t S_max;
    uint64_t *gt_col;                                     // [NP] genotype key of each DP column (genotype_key, 0 = unknown), null without dosages
    int32_t *path; uint8_t *hap_allele; double *dp_cost;
    // ---- CSR cells out
    int64_t *cell_off; int32_t *cell_pos; uint8_t *cell_allele;
    int64_t cell_base;                                    // cells of the chunks before this one: cell_off is global, cell_pos / cell_allele are local
};

}  // namespace ahs
