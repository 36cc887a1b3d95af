// tests/native/oracle_genotypes.cpp — TEST INFRASTRUCTURE, NOT PRODUCT CODE.
//
// The CPU oracle with caller-supplied genotypes: the rule of ahs_phase_batch_genotyped (include/ahsoka_b200.h), built on
// oracle/phase_oracle.cpp as it is.  Built by __graft_entry__.build() into oracle/_ref/liboracle_gt.so; bound by
// tests/oracle_genotypes.py.
//
// phase_chain() of the oracle threads a chain against the built-in genotypes ({0:1,1:1} at ploidy 2, the empty map =
// "not all consensus alleles equal" above; rule R3 of oracle/core/phase_core.hpp).  This file compiles the oracle with its
// one call of thread_paths() routed through thread_paths_caller_gt(), which puts the caller's genotype map in place of
// genotypes[q] wherever a thread-local table has one.  A chain is phased twice: plainly, which yields its covered
// positions (the bubble ids of its DP columns), then with the table built from the dosages of those bubbles.  Nothing
// before the DP depends on the genotypes, so both passes see the same columns.
#include <unordered_map>
#include <vector>

#include "../../oracle/core/phase_core.hpp"

namespace {
using GenotypeMap = std::unordered_map<uint32_t, uint32_t>;
thread_local const std::vector<GenotypeMap>* g_caller_gt = nullptr;     // [n_pos] of the chain being phased; empty map = unknown
}

inline ahs_oracle::ThreadResult thread_paths_caller_gt(uint32_t ploidy, double switchCost, double affineSwitchCost, uint32_t start,
                                                      uint32_t end, const std::vector<std::vector<uint32_t>>& covMap,
                                                      const std::vector<std::vector<double>>& coverage,
                                                      const std::vector<std::vector<uint32_t>>& consensus,
                                                      const std::vector<GenotypeMap>& genotypes) {
    if (!g_caller_gt) return ahs_oracle::thread_paths(ploidy, switchCost, affineSwitchCost, start, end, covMap, coverage, consensus, genotypes);
    std::vector<GenotypeMap> g = genotypes;
    for (size_t q = 0; q < g_caller_gt->size() && q < g.size(); q++) if (!(*g_caller_gt)[q].empty()) g[q] = (*g_caller_gt)[q];
    return ahs_oracle::thread_paths(ploidy, switchCost, affineSwitchCost, start, end, covMap, coverage, consensus, g);
}

#define thread_paths thread_paths_caller_gt
#include "../../oracle/phase_oracle.cpp"
#undef thread_paths

namespace {

// one chain: the oracle's phase_chain, with the caller's genotype at every covered position whose dosages are known
void phase_chain_gt(const ahs_batch_in* in, const uint8_t* dosage, int c, ChainOut& o) {
    phase_chain(in, c, o);
    if (o.status != AHS_CHAIN_OK) return;
    std::vector<GenotypeMap> gt(o.pos.size());
    bool any = false;
    for (size_t q = 0; q < o.pos.size(); q++) {
        const int64_t gb = in->bubble_off[c] + o.pos[q];
        for (int64_t a = in->allele_off[gb]; a < in->allele_off[gb + 1]; a++)
            if (dosage[a]) gt[q][(uint32_t)(a - in->allele_off[gb])] = dosage[a];
        any |= !gt[q].empty();
    }
    if (!any) return;
    ChainOut with_gt;
    g_caller_gt = &gt;
    phase_chain(in, c, with_gt);
    g_caller_gt = nullptr;
    o = with_gt;
}

}  // namespace

extern "C" {

// ahs_oracle_phase_batch with allele dosages (indexed like allele_off); AHS_ERR_ARG where a bubble's dosages are neither all
// 0 nor sum to the ploidy.  allele_dosage == NULL: ahs_oracle_phase_batch.
int ahs_oracle_phase_batch_gt(const ahs_batch_in* in, const uint8_t* allele_dosage, ahs_batch_out* out, int n_threads) {
    if (!in || !out || in->ploidy < 1) return AHS_ERR_ARG;
    if (!allele_dosage) return ahs_oracle_phase_batch(in, out, n_threads);
    const int C = in->n_chains;
    if (C > 0)
        for (int64_t gb = 0; gb < in->bubble_off[C]; gb++) {
            int sum = 0;
            for (int64_t a = in->allele_off[gb]; a < in->allele_off[gb + 1]; a++) sum += allele_dosage[a];
            if (sum != 0 && sum != in->ploidy) return AHS_ERR_ARG;
        }
    memset(out, 0, sizeof(*out));
    std::vector<ChainOut> co(C);
    {
        int nt = n_threads > 0 ? n_threads : (int)std::thread::hardware_concurrency();
        if (nt < 1) nt = 1;
        if (nt > C) nt = C > 0 ? C : 1;
        std::atomic<int> next(0);
        auto worker = [&]() { for (int c = next.fetch_add(1); c < C; c = next.fetch_add(1)) phase_chain_gt(in, allele_dosage, c, co[c]); };
        if (nt == 1) worker();
        else { std::vector<std::thread> th; for (int t = 0; t < nt; t++) th.emplace_back(worker); for (auto& t : th) t.join(); }
    }
    // packed exactly as ahs_oracle_phase_batch packs its chains
    std::vector<int32_t> status, read_id, read_mapq, read_cluster, cell_pos, n_clusters, pos, path, maxpos;
    std::vector<int64_t> read_off{0}, cell_off{0}, pos_off{0};
    std::vector<uint8_t> cell_allele, hap_allele; std::vector<double> dp_cost;
    int64_t n_pairs = 0, n_ok = 0;
    for (int c = 0; c < C; c++) {
        ChainOut& o = co[c];
        status.push_back(o.status); n_clusters.push_back(o.n_clusters); dp_cost.push_back(o.dp_cost); maxpos.push_back(o.maxpos);
        read_id.insert(read_id.end(), o.read_id.begin(), o.read_id.end());
        read_mapq.insert(read_mapq.end(), o.read_mapq.begin(), o.read_mapq.end());
        read_cluster.insert(read_cluster.end(), o.read_cluster.begin(), o.read_cluster.end());
        for (int64_t n : o.cell_cnt) cell_off.push_back(cell_off.back() + n);
        cell_pos.insert(cell_pos.end(), o.cell_pos.begin(), o.cell_pos.end());
        cell_allele.insert(cell_allele.end(), o.cell_allele.begin(), o.cell_allele.end());
        pos.insert(pos.end(), o.pos.begin(), o.pos.end());
        path.insert(path.end(), o.path.begin(), o.path.end());
        hap_allele.insert(hap_allele.end(), o.hap_allele.begin(), o.hap_allele.end());
        read_off.push_back((int64_t)read_id.size()); pos_off.push_back((int64_t)pos.size());
        n_pairs += o.n_pairs; if (o.status == AHS_CHAIN_OK) n_ok++;
    }
    out->n_chains = C; out->ploidy = in->ploidy;
    out->status = dup(status); out->read_off = dup(read_off); out->read_id = dup(read_id); out->read_mapq = dup(read_mapq);
    out->read_cluster = dup(read_cluster); out->cell_off = dup(cell_off); out->cell_pos = dup(cell_pos); out->cell_allele = dup(cell_allele);
    out->n_clusters = dup(n_clusters); out->pos_off = dup(pos_off); out->pos = dup(pos); out->path = dup(path);
    out->hap_allele = dup(hap_allele); out->dp_cost = dup(dp_cost); out->maxpos = dup(maxpos);
    out->n_cells = (int64_t)cell_pos.size(); out->n_pairs = n_pairs; out->n_chains_ok = n_ok;
    return AHS_OK;
}

}  // extern "C"
